// engine.cu — host side of the B200 reconstruction engine (b200hevc.h part 2) + kernel launches.
//
// Per picture: validate the records, build the work lists (MC units, k_residual classes, intra tasks in topological
// order) and pack everything into one pinned staging buffer on a small host thread pool, ONE host->device copy, then
//   k_inter_pred_tma -> k_residual -> k_mark_pending + k_intra -> k_deblock<V> -> k_deblock<H> -> k_sao8 (or k_sao_prep + k_sao)
// on one of the engine's streams; pictures are pipelined over the streams with per-slot event ordering.
// Reference pictures never leave the device (DPB slots are device surfaces).
// There is no CPU fallback: without a CUDA device b200_engine_create fails with B200_ERR_NO_DEVICE.

#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <exception>
#include <functional>
#include <mutex>
#include <string>
#include <sched.h>
#include <thread>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "b200hevc.h"
#include "dev_common.cuh"
#include "kernels_filter.cuh"
#include "kernels_mc.cuh"
#include "kernels_mc8.cuh"
#include "kernels_mct.cuh"
#include "kernels_recon.cuh"

// ---- error reporting -----------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static int set_err(int code, const char* fmt, ...)
{
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
extern "C" const char* b200_last_error(void) { return g_err; }

#define CU(call)                                                                                        \
  do {                                                                                                  \
    cudaError_t e_ = (call);                                                                            \
    if (e_ != cudaSuccess) return set_err(B200_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---- surfaces ------------------------------------------------------------------------------------
// A surface keeps a replicated BORDER around every plane (B200_PAD_* samples on each side) so that the motion-compensation
// kernel never clamps a coordinate: mc_luma / mc_chroma clamp every reference sample position to the picture
// (motion.cc:147-153, 251-254), which is the same as reading a picture whose edge samples are replicated outwards; a window
// that lies further out than the border is moved to the border's rim, where every sample already is the edge sample.
// plane[c] points at sample (0, 0); the two chroma planes share one allocation (fixed plane stride) so that one 3-D TMA box
// fetches the Cb and the Cr window of a prediction unit.
// (B200_PAD_X / _Y / _CX / _CY: dev_common.cuh)

struct Surface {
  uint8_t* plane[3] = {nullptr, nullptr, nullptr};  // sample (0,0) of each plane
  uint8_t* alloc[2] = {nullptr, nullptr};           // luma allocation, chroma allocation (Cb then Cr)
  size_t alloc_bytes[2] = {0, 0};
  int pitch[3] = {0, 0, 0};
  int w = 0, h = 0, cw = 0, ch = 0, chroma = 0, bd_y = 0, bd_c = 0;
  bool valid = false;  // holds a picture
  bool has_tm = false; // tensor maps of the padded planes for the TMA-staged MC kernel (8-bit surfaces)
  CUtensorMap tm_luma[2], tm_chroma[2];  // [0] big boxes, [1] small boxes (kernels_mct.cuh)
};

// cuTensorMapEncodeTiled through the runtime (no link-time dependency on libcuda)
typedef CUresult (*b200_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                         const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static b200_encode_tiled_fn encode_tiled()
{
  static b200_encode_tiled_fn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess) p = nullptr;
    return (b200_encode_tiled_fn)p;
  }();
  return fn;
}

static void surface_free(Surface& s)
{
  for (int i = 0; i < 2; i++) {
    if (s.alloc[i]) cudaFree(s.alloc[i]);
    s.alloc[i] = nullptr;
  }
  for (int c = 0; c < 3; c++) s.plane[c] = nullptr;
  s.w = s.h = 0;
  s.valid = false;
}

static int bytes_per_sample(int bd) { return bd > 8 ? 2 : 1; }

// New surfaces are zero-filled ON THE ENGINE'S STREAM (it is non-blocking: a memset on the legacy stream could land after
// kernels launched later on the engine's stream).
static int surface_ensure(Surface& s, const b200_pic_params& p, cudaStream_t st)
{
  const int cw = p.chroma_format_idc ? p.width / 2 : 0, ch = p.chroma_format_idc ? p.height / 2 : 0;
  if (s.plane[0] && s.w == p.width && s.h == p.height && s.chroma == p.chroma_format_idc &&
      bytes_per_sample(s.bd_y) == bytes_per_sample(p.bit_depth_luma) && bytes_per_sample(s.bd_c) == bytes_per_sample(p.bit_depth_chroma)) {
    s.bd_y = p.bit_depth_luma;
    s.bd_c = p.bit_depth_chroma;
    return B200_OK;
  }
  surface_free(s);
  s.w = p.width; s.h = p.height; s.cw = cw; s.ch = ch; s.chroma = p.chroma_format_idc;
  s.bd_y = p.bit_depth_luma; s.bd_c = p.bit_depth_chroma;
  const int bl = bytes_per_sample(p.bit_depth_luma), bc = bytes_per_sample(p.bit_depth_chroma);
  // rows padded to 256 bytes: sample (0, y) is 128-byte aligned, every CTB row segment 16-byte aligned, and vector accesses may
  // overshoot the picture width inside the border
  s.pitch[0] = (int)align_up((size_t)(p.width + 2 * B200_PAD_X) * bl, 256);
  s.pitch[1] = s.pitch[2] = cw ? (int)align_up((size_t)(cw + 2 * B200_PAD_CX) * bc, 256) : 0;
  s.alloc_bytes[0] = (size_t)s.pitch[0] * (p.height + 2 * B200_PAD_Y);
  CU(cudaMalloc(&s.alloc[0], s.alloc_bytes[0]));
  CU(cudaMemsetAsync(s.alloc[0], 0, s.alloc_bytes[0], st));
  s.plane[0] = s.alloc[0] + (size_t)B200_PAD_Y * s.pitch[0] + (size_t)B200_PAD_X * bl;
  if (cw) {
    const size_t plane_bytes = (size_t)s.pitch[1] * (ch + 2 * B200_PAD_CY);
    s.alloc_bytes[1] = 2 * plane_bytes;
    CU(cudaMalloc(&s.alloc[1], s.alloc_bytes[1]));
    CU(cudaMemsetAsync(s.alloc[1], 0, s.alloc_bytes[1], st));
    for (int c = 1; c < 3; c++) s.plane[c] = s.alloc[1] + (c - 1) * plane_bytes + (size_t)B200_PAD_CY * s.pitch[1] + (size_t)B200_PAD_CX * bc;
  }
  s.has_tm = false;
  if (bl == 1 && bc == 1) {
    // Tensor maps over the PADDED planes (coordinate = picture coordinate + border): rows of `pitch` bytes; boxes of one MC
    // tile's reference window (kernels_mct.cuh).  Out-of-range box parts (skew rows above the surface) are zero-filled and unused.
    b200_encode_tiled_fn enc = encode_tiled();
    if (!enc) return set_err(B200_ERR_CUDA, "cuTensorMapEncodeTiled unavailable");
    for (int k = 0; k < 2; k++) {
      cuuint64_t dims[2] = {(cuuint64_t)s.pitch[0], (cuuint64_t)(p.height + 2 * B200_PAD_Y)}, strides[1] = {(cuuint64_t)s.pitch[0]};
      cuuint32_t box[2] = {(cuuint32_t)(k ? MCT_LWS_PITCH : MCT_LWB_PITCH), (cuuint32_t)(k ? MCT_LWS_ROWS : MCT_LWB_ROWS)}, es[2] = {1, 1};
      if (enc(&s.tm_luma[k], CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, s.alloc[0], dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
              CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return set_err(B200_ERR_CUDA, "cuTensorMapEncodeTiled (luma) failed");
      if (cw) {
        cuuint64_t cdims[3] = {(cuuint64_t)s.pitch[1], (cuuint64_t)(ch + 2 * B200_PAD_CY), 2};
        cuuint64_t cstrides[2] = {(cuuint64_t)s.pitch[1], (cuuint64_t)s.pitch[1] * (ch + 2 * B200_PAD_CY)};
        cuuint32_t cbox[3] = {(cuuint32_t)(k ? MCT_CWS_PITCH : MCT_CWB_PITCH), (cuuint32_t)(k ? MCT_CWS_ROWS : MCT_CWB_ROWS), 2}, ces[3] = {1, 1, 1};
        if (enc(&s.tm_chroma[k], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, s.alloc[1], cdims, cstrides, cbox, ces, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
          return set_err(B200_ERR_CUDA, "cuTensorMapEncodeTiled (chroma) failed");
      } else {
        s.tm_chroma[k] = s.tm_luma[k];
      }
    }
    s.has_tm = true;
  }
  return B200_OK;
}

// Replicates the edge samples of a finished picture into its border (one launch for all planes).  blockIdx.y = plane.
//   part 1 (rows 0..h-1): the pad_x samples left of column 0 and right of column w-1;
//   part 2 (pad_y rows above row 0 and below row h-1): the whole padded row, copied from row 0 / h-1 with the column clamped.
template <typename P>
__global__ void k_extend_borders(uint8_t* p0, uint8_t* p1, uint8_t* p2, int pitch0, int pitch1, int w, int h, int cw, int ch)
{
  const int c = blockIdx.y;
  uint8_t* base = c == 0 ? p0 : c == 1 ? p1 : p2;
  const int pitch = c ? pitch1 : pitch0, pw = c ? cw : w, ph = c ? ch : h;
  const int padx = c ? B200_PAD_CX : B200_PAD_X, pady = c ? B200_PAD_CY : B200_PAD_Y;
  constexpr int V = 16 / sizeof(P);       // samples per 16-byte store
  const int side_chunks = padx / V;       // per side and row
  const int n1 = ph * 2 * side_chunks;
  const int row_chunks = (pw + 2 * padx + V - 1) / V;  // the last chunk may overshoot into the row's alignment padding (pitch is a multiple of 256)
  const int n2 = 2 * pady * row_chunks;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n1 + n2; i += gridDim.x * blockDim.x) {
    if (i < n1) {
      const int y = i / (2 * side_chunks), k = i - y * 2 * side_chunks;
      const bool right = k >= side_chunks;
      P* row = row_ptr<P>(base, pitch, y);
      const P v = right ? row[pw - 1] : row[0];
      P* dst = right ? row + pw + (k - side_chunks) * V : row - padx + k * V;
      P tmp[V];
#pragma unroll
      for (int j = 0; j < V; j++) tmp[j] = v;
      if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(tmp);
      else
        for (int j = 0; j < V; j++) dst[j] = v;  // chroma widths that are not a multiple of 16 bytes
    } else {
      const int j2 = i - n1;
      const int r = j2 / row_chunks, k = j2 - r * row_chunks;
      const bool below = r >= pady;
      const int y = below ? ph + (r - pady) : r - pady;
      const P* src = row_ptr<P>(base, pitch, below ? ph - 1 : 0);
      P* dst = row_ptr<P>(base, pitch, y) - padx + k * V;
      const int x0 = k * V - padx;
      P tmp[V];
#pragma unroll
      for (int j = 0; j < V; j++) tmp[j] = src[min(max(x0 + j, 0), pw - 1)];
      *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(tmp);
    }
  }
}

static void launch_extend_borders(const Surface& s, cudaStream_t st)
{
  dim3 grid(148 * 2, s.chroma ? 3 : 1);
  if (bytes_per_sample(s.bd_y) == 2)
    k_extend_borders<uint16_t><<<grid, 256, 0, st>>>(s.plane[0], s.plane[1], s.plane[2], s.pitch[0], s.pitch[1], s.w, s.h, s.cw, s.ch);
  else
    k_extend_borders<uint8_t><<<grid, 256, 0, st>>>(s.plane[0], s.plane[1], s.plane[2], s.pitch[0], s.pitch[1], s.w, s.h, s.cw, s.ch);
}

// ---- engine --------------------------------------------------------------------------------------
struct StagingSet {
  uint8_t* host = nullptr;  // pinned
  uint8_t* dev = nullptr;
  size_t cap = 0;
  cudaEvent_t done = nullptr;  // recorded after the last kernel that reads `dev`
  bool in_flight = false;
  std::atomic<size_t>* cap_hint = nullptr;  // the owning engine's largest capacity so far (ensure_staging)
};

// A few host threads for the per-picture host work (validation / work-list building of the PUs next to that of the TUs,
// copying the record arrays into the pinned staging buffer): submit_picture is host-bound on large pictures otherwise.
struct HostPool {
  // Jobs belong to a group; wait(group) returns when that group's jobs are done, so several threads (the asynchronous planners)
  // can share one pool.
  struct Group { int pending = 0; };
  std::vector<std::thread> th;
  std::mutex m;
  std::condition_variable cv, done_cv;
  std::deque<std::pair<Group*, std::function<void()>>> q;
  Group own;
  bool stop = false;
  void start(int n)
  {
    for (int i = 0; i < n; i++)
      th.emplace_back([this] {
        for (;;) {
          std::pair<Group*, std::function<void()>> job;
          {
            std::unique_lock<std::mutex> lk(m);
            cv.wait(lk, [this] { return stop || !q.empty(); });
            if (stop && q.empty()) return;
            job = std::move(q.front());
            q.pop_front();
          }
          job.second();
          {
            std::lock_guard<std::mutex> lk(m);
            if (--job.first->pending == 0) done_cv.notify_all();
          }
        }
      });
  }
  void run(Group* g, std::function<void()> f)
  {
    if (th.empty()) { f(); return; }
    {
      std::lock_guard<std::mutex> lk(m);
      q.emplace_back(g, std::move(f));
      g->pending++;
    }
    cv.notify_one();
  }
  void wait(Group* g)
  {
    std::unique_lock<std::mutex> lk(m);
    done_cv.wait(lk, [g] { return g->pending == 0; });
  }
  void run(std::function<void()> f) { run(&own, std::move(f)); }
  void wait() { wait(&own); }
  ~HostPool()
  {
    {
      std::lock_guard<std::mutex> lk(m);
      stop = true;
    }
    cv.notify_all();
    for (auto& t : th) t.join();
  }
};

// One pipeline context = one CUDA stream with everything a picture in flight needs privately.  Pictures are placed on the
// contexts by pick_ctx; cross-context ordering comes from per-slot events (SlotSync): a picture waits for the
// writers of its reference slots and for every earlier reader / writer of its destination slot.  So pictures that do
// not depend on each other (the B pictures of one hierarchy level, the next intra period's I picture) overlap, and a
// latency-bound kernel (the intra DAG) of one picture leaves the SMs to the others.
#define B200_MAX_CTX 12
#define B200_MAX_PHYS (B200_MAX_SLOTS + 32)  // physical surfaces: every name plus the renamed pictures in flight
#define B200_STAGE_SETS 40
struct PipeCtx {
  cudaStream_t stream = nullptr;
  Surface scratch;              // pre-SAO picture
  uint8_t* sync_buf = nullptr;  // [256 B ticket | pending map Y | Cb | Cr | SAO masks]
  size_t sync_cap = 0;
  cudaEvent_t tail = nullptr;   // b200_engine_join
};

struct SlotSync {
  cudaEvent_t written = nullptr;
  int writer = -1;                       // context of the last writer, -1: none in flight
  cudaEvent_t read[B200_MAX_CTX] = {};   // last read of this slot issued on each context
  bool read_pending[B200_MAX_CTX] = {};
};

#define PLAN_PU_PARTS 4
#define PLAN_INTRA_PARTS 8
struct IntraPart {
  uint32_t i0 = 0, i1 = 0, task_base = 0;
  std::vector<uint32_t> intra_idx, task_of, task_cell, fill;  // task_cell: region cell x | y << 12 | cells per side << 24 | plane << 28
};

struct AsyncState;
struct b200_engine {
  int device = 0;
  std::atomic<size_t> stage_cap_hint{0};
  std::mutex issue_m;  // held by the asynchronous sequencer while it issues a command (it mutates the slot / stream state b200_engine_wait_slot reads)
  AsyncState* async = nullptr;  // b200_engine_submit_picture_async: planner threads + the in-order sequencer (created on first use)
  PipeCtx ctx[B200_MAX_CTX];
  // Record staging: pinned host buffer + device arena per picture in flight, handed out round-robin whatever stream the picture
  // runs on (a set is reused when the kernels of the picture that used it B200_STAGE_SETS pictures ago have finished)
  StagingSet stage_pool[B200_STAGE_SETS];
  unsigned next_stage = 0;
  int n_ctx = 1;
  // DPB slots are NAMES (what the records' ref_slot / dst_slot say); the pictures live in a pool of physical surfaces.  A picture
  // that writes slot d while earlier pictures on other streams still read (or write) d's current surface gets another, idle
  // surface and the name moves — like register renaming, WAR / WAW hazards between pictures cost nothing, whatever slot policy
  // the host's DPB has (libde265 reuses the first free image, dpb.cc: the hazard is the common case).  Only true (RAW)
  // dependencies remain.
  Surface slot[B200_MAX_PHYS];
  SlotSync ssync[B200_MAX_PHYS];
  int lmap[B200_MAX_SLOTS];       // name -> physical surface, -1: never written
  int owner[B200_MAX_PHYS];       // physical surface -> name it currently carries, -1: free (may still have readers in flight)
  int last_owner[B200_MAX_PHYS];  // the name it carried last (b200_engine_wait_slot also waits for reads of a renamed-away surface)
  uint64_t pool_geom = 0;  // format of the last picture issued (run_layout)
  uint64_t n_renamed = 0;
  b200_engine()
  {
    for (int& v : lmap) v = -1;
    for (int& v : owner) v = -1;
    for (int& v : last_owner) v = -1;
  }
  HostPool pool;
  // A shadow engine (asynchronous planner) plans a picture on its own thread; for a picture with a long plan (a large intra
  // picture) it borrows the owning engine's pool so that the in-order sequencer is not held up by it.
  HostPool* helper = nullptr;
  HostPool::Group helper_group;
  bool use_helper = false;
  void prun(std::function<void()> f)
  {
    if (use_helper) helper->run(&helper_group, std::move(f));
    else pool.run(std::move(f));
  }
  void pwait()
  {
    if (use_helper) helper->wait(&helper_group);
    else pool.wait();
  }
  int num_sms = 148;
  long long slot_depth[B200_MAX_SLOTS] = {}, tail_depth[B200_MAX_CTX] = {}, key_depth = 0;  // pick_ctx: dependency depths
  int n_ind = 2, next_ind = 0, ind_run = 0;  // streams for pictures that read no reference (intra pictures), used round-robin (B200_IND_STREAMS)
  int intra_i_grid = 64;        // grid cap of k_intra for such pictures: the DAG is at most ~160 tasks wide, 64 CTAs (512 warps) cover it and leave the other SMs to the P/B pictures (0: one CTA per SM; B200_INTRA_I_GRID)
  unsigned int *intra_err = nullptr, *intra_err_host = nullptr;  // k_intra gave up a dependency wait (device word; mapped host copy)
  unsigned long long spin_limit_ns = 2000000000ull;              // B200_INTRA_SPIN_LIMIT_MS
  int intra_ctas = 3, poll_ns = 256;  // k_intra: persistent CTAs per SM, back-off cap of the flag polling (B200_INTRA_CTAS / B200_POLL_NS)
  // B200_TIMELINE=<file>: a CUDA event before and after every launch; the intervals of all streams (ms since the first launch)
  // are appended to the file at b200_engine_sync / destroy: which kernels of which pictures really overlap (tools/timeline.py)
  struct TlEntry { cudaEvent_t e0, e1; const char* name; int poc, ctx; };
  std::vector<TlEntry> tl;
  const char* tl_path = nullptr;
  cudaEvent_t tl_base = nullptr;
  int mc_ctas = 3;        // k_inter_pred_tma: persistent CTAs per SM (B200_MC_CTAS)
  bool timing = false;
  std::vector<cudaEvent_t> tev;  // timing ring: TIMING_RING pictures x 7 events
  unsigned tcount = 0;           // pictures recorded since enable / reset
  cudaEvent_t* ev = nullptr;     // events of the picture being submitted
  uint64_t launches = 0;
  double host_s[4] = {0, 0, 0, 0};  // submit_picture host time: [0] validate + staging wait, [1] plan + pack, [3] launches (B200_HOST_PROF=1 prints at destroy)
  uint64_t host_n = 0;
  // asynchronous path, same switch: [0] planner busy (sum over threads), [1] sequencer waiting for a plan, [2] sequencer issuing pictures,
  // [3] sequencer issuing read-backs; run_layout segments: [4] surfaces + H2D copy, [5] order_before, [6] kernels, [7] border + order_after
  double async_s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  uint64_t async_n = 0;
  bool host_prof = false;
  int host_skip = 0;
  // host scratch reused across pictures
  std::vector<uint32_t> part_a[8][3];  // plan_intra_A: per range, per k_residual class
  std::vector<uint32_t> pu_tiles[PLAN_PU_PARTS];  // plan_pus_part
  size_t pu_count[PLAN_PU_PARTS][8] = {};
  uint32_t pu_ref_mask[PLAN_PU_PARTS] = {};
  IntraPart ipart[PLAN_INTRA_PARTS];              // plan_intra_*
  std::vector<uint32_t> cell_level[3], task_level, level_off;  // plan_intra_levels
  std::vector<uint32_t> ctb_count, tiles, tiles_sorted, list_a, list_b, intra_idx, task_of, task_first, task_start, task_order;
};

static int async_flush(b200_engine* en);
static void async_stop(b200_engine* en);

#define TIMING_RING 256

static void tl_begin(b200_engine* en, cudaStream_t st, const char* name, int poc, int ctx)
{
  b200_engine::TlEntry e{nullptr, nullptr, name, poc, ctx};
  cudaEventCreate(&e.e0);
  cudaEventCreate(&e.e1);
  if (!en->tl_base) { cudaEventCreate(&en->tl_base); cudaEventRecord(en->tl_base, st); }
  cudaEventRecord(e.e0, st);
  en->tl.push_back(e);
}
static void tl_end(b200_engine* en, cudaStream_t st) { cudaEventRecord(en->tl.back().e1, st); }
static void tl_flush(b200_engine* en)  // after all streams were synchronised
{
  if (!en->tl_path || en->tl.empty()) return;
  if (FILE* f = fopen(en->tl_path, "a")) {
    for (auto& e : en->tl) {
      float t0 = 0, t1 = 0;
      cudaEventElapsedTime(&t0, en->tl_base, e.e0);
      cudaEventElapsedTime(&t1, en->tl_base, e.e1);
      fprintf(f, "%d %s %d %.4f %.4f\n", e.ctx, e.name, e.poc, t0, t1);
    }
    fclose(f);
  }
  for (auto& e : en->tl) { cudaEventDestroy(e.e0); cudaEventDestroy(e.e1); }
  en->tl.clear();
}
#define TL(name, launch)                                                              \
  do {                                                                                \
    if (en->tl_path) tl_begin(en, st, name, L.params.poc, (int)(&cx - en->ctx));      \
    launch;                                                                           \
    if (en->tl_path) tl_end(en, st);                                                  \
  } while (0)

struct PicLayout {
  size_t off[14] = {}, total = 0, raw_total = 0, unit_cap = 0;
  uint32_t ref_mask = 0;  // slots the picture's PUs read
  int n_tiles = 0, n_batches = 0, n_a = 0, n_aw = 0, n_a8 = 0, n_b = 0, n_task = 0;
  bool direct = false;                   // B200_PIC_RECORDS_PINNED: raw sections are uploaded from raw_src (the caller's arrays)
  const void* raw_src[14] = {};
  size_t raw_sz[14] = {};
  int intra_levels = 0, intra_width = 0;  // intra DAG: number of levels, tasks in the widest level (B200_HOST_PROF prints them)
  bool run_deblock = false, run_sao = false, has_scaling = false;
  b200_pic_params params{};
  uint32_t n_tu = 0;
};

struct b200_prepared {
  uint8_t* dev = nullptr;
  PicLayout L;
};

static bool g_tables_ready[64] = {};

static int init_tables(int device)
{
  if (device < 64 && g_tables_ready[device]) return B200_OK;
  // HEVC core transform: mat[k][n] = +-T((2n+1)k mod 128) with T = first matrix column (cosine symmetry);
  // the 32 base magnitudes are the transform's definition (fallback-dct.cc:512-545 column 0).
  static const int8_t T[33] = {64, 90, 90, 90, 89, 88, 87, 85, 83, 82, 80, 78, 75, 73, 70, 67, 64,
                               61, 57, 54, 50, 46, 43, 38, 36, 31, 25, 22, 18, 13, 9,  4,  0};
  int8_t m[32][32];
  for (int k = 0; k < 32; k++)
    for (int n = 0; n < 32; n++) {
      int j = ((2 * n + 1) * k) % 128, sign = 1;
      if (j > 64) j = 128 - j;
      if (j > 32) { j = 64 - j; sign = -1; }
      m[k][n] = (int8_t)(sign * T[j]);
    }
  CU(cudaMemcpyToSymbol(c_dct, m, sizeof(m)));
  {  // packed transform matrices of the sub-warp residual paths (kernels_residual.cuh): 4 rows of one column per word
    static ResTables rt;
    auto col4 = [&](int nT, int jq, int i) {
      uint32_t w = 0;
      for (int b = 0; b < 4; b++) w |= (uint32_t)(uint8_t)m[(32 / nT) * (4 * jq + b)][i] << (8 * b);
      return w;
    };
    for (int i = 0; i < 4; i++) rt.m4[i] = col4(4, 0, i);
    for (int jq = 0; jq < 2; jq++) for (int i = 0; i < 8; i++) rt.m8[jq][i] = col4(8, jq, i);
    for (int jq = 0; jq < 4; jq++) for (int i = 0; i < 16; i++) rt.m16[jq][i] = col4(16, jq, i);
    for (int jq = 0; jq < 8; jq++) for (int i = 0; i < 32; i++) rt.m32[jq][i] = col4(32, jq, i);
    // DST-VII: M[j][i] = round(128 * 2/3 * sin((2j+1)(i+1)pi/9)) (fallback-dct.cc:260-265 holds the same 16 numbers)
    for (int i = 0; i < 4; i++) {
      uint32_t w = 0;
      for (int j = 0; j < 4; j++) w |= (uint32_t)(uint8_t)(int8_t)lround(128.0 * 2.0 / 3.0 * sin((2 * j + 1) * (i + 1) * M_PI / 9.0)) << (8 * j);
      rt.dst4[i] = w;
    }
    CU(cudaMemcpyToSymbol(c_res, &rt, sizeof(rt)));
  }
  {  // packed tap tables of the 8-bit MC kernels (kernels_mc8.cuh mc8_build_tables)
    static Mc8Tables tb;
    mc8_build_tables(tb);
    CU(cudaMemcpyToSymbol(c_mc8, &tb, sizeof(tb)));
  }
  if (device < 64) g_tables_ready[device] = true;
  return B200_OK;
}

extern "C" int b200_engine_create(b200_engine** out, int device)
{
  if (!out) return set_err(B200_ERR_INVALID, "null out");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return set_err(B200_ERR_NO_DEVICE, "no CUDA device available (%s); the B200 engine has no CPU fallback", cudaGetErrorString(e));
  if (device < 0 || device >= n) return set_err(B200_ERR_INVALID, "device %d out of range (0..%d)", device, n - 1);
  CU(cudaSetDevice(device));
  b200_engine* en = new (std::nothrow) b200_engine();
  if (!en) return set_err(B200_ERR_NOMEM, "out of memory");
  en->device = device;
  int rc = init_tables(device);
  if (rc) { delete en; return rc; }
  en->n_ctx = 8;
  {
    int nt = 8;
    if (const char* e = getenv("B200_HOST_THREADS")) nt = std::max(0, std::min(16, atoi(e)));
    en->pool.start(nt);
  }
  if (const char* e = getenv("B200_INTRA_CTAS")) en->intra_ctas = std::max(1, std::min(4, atoi(e)));
  if (const char* e = getenv("B200_IND_STREAMS")) en->n_ind = std::max(1, std::min(4, atoi(e)));
  if (const char* e = getenv("B200_INTRA_I_GRID")) en->intra_i_grid = std::max(0, atoi(e));
  if (const char* e = getenv("B200_POLL_NS")) en->poll_ns = std::max(32, std::min(100000, atoi(e)));
  if (const char* e = getenv("B200_INTRA_SPIN_LIMIT_MS")) en->spin_limit_ns = 1000000ull * (unsigned long long)std::max(1, std::min(60000, atoi(e)));
  en->tl_path = getenv("B200_TIMELINE");
  en->host_prof = getenv("B200_HOST_PROF") != nullptr;
  if (const char* e = getenv("B200_HOST_PROF_SKIP")) en->host_skip = std::max(0, atoi(e));
  if (const char* e = getenv("B200_MC_CTAS")) en->mc_ctas = std::max(1, std::min(8, atoi(e)));
  if (const char* e = getenv("B200_STREAMS")) en->n_ctx = std::max(1, std::min(B200_MAX_CTX, atoi(e)));
  for (int k = 0; k < B200_MAX_CTX; k++) {
    PipeCtx& cx = en->ctx[k];
    CU(cudaStreamCreateWithFlags(&cx.stream, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&cx.tail, cudaEventDisableTiming));
  }
  for (auto& st : en->stage_pool) {
    CU(cudaEventCreateWithFlags(&st.done, cudaEventDisableTiming | cudaEventBlockingSync));
    st.cap_hint = &en->stage_cap_hint;
  }  // planner threads sleep, not spin, on a busy set
  CU(cudaMalloc(&en->intra_err, 256));
  CU(cudaMemset(en->intra_err, 0, 256));
  CU(cudaHostAlloc(&en->intra_err_host, 64, cudaHostAllocMapped));
  *en->intra_err_host = 0;
  for (auto& ss : en->ssync) {
    CU(cudaEventCreateWithFlags(&ss.written, cudaEventDisableTiming));
    for (int k = 0; k < B200_MAX_CTX; k++) CU(cudaEventCreateWithFlags(&ss.read[k], cudaEventDisableTiming));
  }
  CU(cudaFuncSetAttribute(k_inter_pred_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(MctShared)));
  CU(cudaFuncSetAttribute(k_intra<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IntraSmem<uint8_t>)));
  CU(cudaFuncSetAttribute(k_intra<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IntraSmem<uint16_t>)));
  CU(cudaDeviceGetAttribute(&en->num_sms, cudaDevAttrMultiProcessorCount, device));
  *out = en;
  return B200_OK;
}

extern "C" void b200_engine_destroy(b200_engine* en)
{
  if (!en) return;
  cudaSetDevice(en->device);
  async_stop(en);
  cudaDeviceSynchronize();
  tl_flush(en);
  if (en->tl_base) cudaEventDestroy(en->tl_base);
  if (getenv("B200_HOST_PROF")) {
    int n_surf = 0;
    for (const auto& sf : en->slot) n_surf += sf.plane[0] != nullptr;
    fprintf(stderr, "[b200] %llu pictures took their destination name to another surface (slot renaming); %d surfaces allocated\n",
            (unsigned long long)en->n_renamed, n_surf);
  }
  if (getenv("B200_HOST_PROF") && en->async_n)
    fprintf(stderr, "[b200] submit_picture_async host ms/picture over %llu pictures: planner busy (all threads) %.3f | sequencer: waiting for a plan %.3f  "
            "pictures %.3f (surfaces+H2D %.3f  order_before %.3f  kernels %.3f  borders+order_after %.3f)  read-backs %.3f\n",
            (unsigned long long)en->async_n, 1e3 * en->async_s[0] / en->async_n, 1e3 * en->async_s[1] / en->async_n, 1e3 * en->async_s[2] / en->async_n,
            1e3 * en->async_s[4] / en->async_n, 1e3 * en->async_s[5] / en->async_n, 1e3 * en->async_s[6] / en->async_n, 1e3 * en->async_s[7] / en->async_n,
            1e3 * en->async_s[3] / en->async_n);
  if (getenv("B200_HOST_PROF") && en->host_n)
    fprintf(stderr, "[b200] submit_picture host ms/picture over %llu pictures: validate+staging-wait %.3f  plan+pack (threaded) %.3f  launch %.3f\n",
            (unsigned long long)en->host_n, 1e3 * en->host_s[0] / en->host_n, 1e3 * en->host_s[1] / en->host_n, 1e3 * en->host_s[3] / en->host_n);
  for (auto& s : en->slot) surface_free(s);
  for (auto& cx : en->ctx) {
    surface_free(cx.scratch);
    if (cx.sync_buf) cudaFree(cx.sync_buf);
    if (cx.tail) cudaEventDestroy(cx.tail);
    if (cx.stream) cudaStreamDestroy(cx.stream);
  }
  for (auto& st : en->stage_pool) {
    if (st.host) cudaFreeHost(st.host);
    if (st.dev) cudaFree(st.dev);
    if (st.done) cudaEventDestroy(st.done);
  }
  for (auto& ss : en->ssync) {
    if (ss.written) cudaEventDestroy(ss.written);
    for (auto& e : ss.read)
      if (e) cudaEventDestroy(e);
  }
  for (auto& e : en->tev)
    if (e) cudaEventDestroy(e);
  if (en->intra_err) cudaFree(en->intra_err);
  if (en->intra_err_host) cudaFreeHost(en->intra_err_host);
  delete en;
}

extern "C" void* b200_engine_stream(b200_engine* en) { return en ? (void*)en->ctx[0].stream : nullptr; }

// After a synchronisation point: did k_intra give up a dependency wait (ReconArgs::err)?  Reported once, then cleared.
static int check_intra_err(b200_engine* en)
{
  if (!en->intra_err_host || !*(volatile unsigned int*)en->intra_err_host) return B200_OK;
  const unsigned int t = *(volatile unsigned int*)en->intra_err_host - 1;
  for (int k = 0; k < B200_MAX_CTX; k++) cudaStreamSynchronize(en->ctx[k].stream);
  *(volatile unsigned int*)en->intra_err_host = 0;
  cudaMemset(en->intra_err, 0, sizeof(unsigned int));
  return set_err(B200_ERR_INVALID, "intra task %u: a neighbour named by the avail bits is never reconstructed before it (dependency wait gave up); picture damaged", t);
}

static int sync_all(b200_engine* en)
{
  for (int k = 0; k < B200_MAX_CTX; k++) CU(cudaStreamSynchronize(en->ctx[k].stream));
  tl_flush(en);
  for (auto& ss : en->ssync) {
    ss.writer = -1;
    for (auto& r : ss.read_pending) r = false;
  }
  return check_intra_err(en);
}

extern "C" int b200_engine_set_streams(b200_engine* en, int n)
{
  if (!en || n < 1 || n > B200_MAX_CTX) return set_err(B200_ERR_INVALID, "stream count must be 1..%d", B200_MAX_CTX);
  CU(cudaSetDevice(en->device));
  { const int frc = async_flush(en); if (frc) return frc; }
  int rc = sync_all(en);
  if (rc) return rc;
  en->n_ctx = n;
  en->next_ind = 0;
  return B200_OK;
}

// Makes stream 0 (b200_engine_stream) wait for everything issued so far on the other streams: an event recorded on
// stream 0 afterwards marks the completion of all submitted pictures.
extern "C" int b200_engine_join(b200_engine* en)
{
  if (!en) return set_err(B200_ERR_INVALID, "null engine");
  CU(cudaSetDevice(en->device));
  { const int frc = async_flush(en); if (frc) return frc; }
  for (int k = 1; k < B200_MAX_CTX; k++) {
    CU(cudaEventRecord(en->ctx[k].tail, en->ctx[k].stream));
    CU(cudaStreamWaitEvent(en->ctx[0].stream, en->ctx[k].tail, 0));
  }
  return B200_OK;
}
extern "C" uint64_t b200_engine_launch_count(const b200_engine* en) { return en ? en->launches : 0; }

extern "C" int b200_engine_enable_timing(b200_engine* en, int on)
{
  if (!en) return set_err(B200_ERR_INVALID, "null engine");
  CU(cudaSetDevice(en->device));
  if (on && en->tev.empty()) {
    en->tev.assign((size_t)TIMING_RING * 7, nullptr);
    for (auto& e : en->tev) CU(cudaEventCreate(&e));
  }
  en->timing = on != 0;
  en->tcount = 0;
  return B200_OK;
}

static int timing_of(b200_engine* en, unsigned idx, float ms[6])
{
  cudaEvent_t* ev = &en->tev[(size_t)(idx % TIMING_RING) * 7];
  CU(cudaEventSynchronize(ev[6]));
  for (int i = 0; i < 5; i++) CU(cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]));
  CU(cudaEventElapsedTime(&ms[5], ev[0], ev[6]));
  return B200_OK;
}

extern "C" int b200_engine_last_timing(b200_engine* en, float ms[6])
{
  if (!en || !ms) return set_err(B200_ERR_INVALID, "null argument");
  if (!en->timing || en->tcount == 0) return set_err(B200_ERR_INVALID, "no timed picture yet");
  CU(cudaSetDevice(en->device));
  return timing_of(en, en->tcount - 1, ms);
}

extern "C" int b200_engine_timing_sum(b200_engine* en, float ms[6], int* n_pictures, int reset)
{
  if (!en || !ms || !n_pictures) return set_err(B200_ERR_INVALID, "null argument");
  CU(cudaSetDevice(en->device));
  for (int i = 0; i < 6; i++) ms[i] = 0;
  const unsigned n = en->timing ? (en->tcount < TIMING_RING ? en->tcount : TIMING_RING) : 0;
  for (unsigned k = 0; k < n; k++) {
    float one[6];
    int rc = timing_of(en, en->tcount - 1 - k, one);
    if (rc) return rc;
    for (int i = 0; i < 6; i++) ms[i] += one[i];
  }
  *n_pictures = (int)n;
  if (reset) en->tcount = 0;
  return B200_OK;
}

static int check_params(const b200_pic_params& p)
{
  if (p.width == 0 || p.height == 0) return set_err(B200_ERR_INVALID, "empty picture");
  if (p.log2_ctb_size < 4 || p.log2_ctb_size > 6) return set_err(B200_ERR_INVALID, "log2_ctb_size %d", p.log2_ctb_size);
  if (p.dst_slot >= B200_MAX_SLOTS) return set_err(B200_ERR_INVALID, "dst_slot %d", p.dst_slot);
  if (p.chroma_format_idc > 1) return set_err(B200_ERR_UNSUPPORTED, "chroma_format_idc %d: the device path implements 4:0:0 and 4:2:0", p.chroma_format_idc);
  if (p.bit_depth_luma < 8 || p.bit_depth_luma > 12 || p.bit_depth_chroma < 8 || p.bit_depth_chroma > 12)
    return set_err(B200_ERR_UNSUPPORTED, "bit depth %d/%d (8..12 supported)", p.bit_depth_luma, p.bit_depth_chroma);
  if ((p.bit_depth_luma > 8) != (p.bit_depth_chroma > 8)) return set_err(B200_ERR_UNSUPPORTED, "mixed 8-bit / high-bit-depth planes");
  if ((p.width & 7) || (p.height & 7)) return set_err(B200_ERR_INVALID, "picture size must be a multiple of the minimum CB size (8)");
  return B200_OK;
}

static DevPic make_devpic(const b200_pic_params& p, const Surface& cur, const Surface& out)
{
  DevPic d{};
  d.w = p.width; d.h = p.height;
  d.cw = cur.cw; d.ch = cur.ch;
  d.bd_y = p.bit_depth_luma; d.bd_c = p.bit_depth_chroma;
  d.log2ctb = p.log2_ctb_size;
  const int S = 1 << d.log2ctb;
  d.wctb = (p.width + S - 1) / S; d.hctb = (p.height + S - 1) / S;
  d.w4 = (p.width + 3) / 4; d.h4 = (p.height + 3) / 4;
  d.w8 = (p.width + 7) / 8; d.h8 = (p.height + 7) / 8;
  d.chroma = p.chroma_format_idc;
  d.cb_qp_off = p.pps_cb_qp_offset; d.cr_qp_off = p.pps_cr_qp_offset;
  d.flags = p.flags;
  for (int c = 0; c < 3; c++) { d.cur[c] = cur.plane[c]; d.out[c] = out.plane[c]; d.pitch[c] = cur.pitch[c]; }
  return d;
}

// sync_buf layout: [256 B ticket | pending map Y | Cb | Cr | (256-aligned) SAO neighbour-availability masks]
static size_t sync_sao_offset(const b200_pic_params& p)
{
  const size_t cw4 = p.chroma_format_idc ? (size_t)((p.width / 2 + 3) / 4) : 0, ch4 = p.chroma_format_idc ? (size_t)((p.height / 2 + 3) / 4) : 0;
  return (256 + (size_t)((p.width + 3) / 4) * ((p.height + 3) / 4) + 2 * cw4 * ch4 + 255) & ~(size_t)255;
}

template <typename P>
static int launch_picture(b200_engine* en, PipeCtx& cx, const PicLayout& L, const DevPic& dp, const RefTable& refs, const uint8_t* dbase)
{
  cudaStream_t st = cx.stream;
  const size_t* off = L.off;
  const int n_tiles = L.n_tiles;
  const bool run_deblock = L.run_deblock, run_sao = L.run_sao;
  if (en->timing) CU(cudaEventRecord(en->ev[1], st));
  if (n_tiles > 0) {
    if (sizeof(P) == 1) {
      // reference windows staged by TMA: the tensor maps of the slots this picture reads travel as a kernel parameter
      MctMaps maps;
      memset(&maps, 0, sizeof(maps));
      int n = 0;
      for (int i = 0; i < B200_MAX_SLOTS; i++) {
        maps.index_of_slot[i] = -1;
        if (!((L.ref_mask >> i) & 1) || !refs.plane[i][0] || !en->slot[en->lmap[i]].has_tm) continue;
        if (n == MCT_MAX_REFS) return set_err(B200_ERR_UNSUPPORTED, "picture references more than %d DPB slots", MCT_MAX_REFS);
        for (int k = 0; k < 2; k++) { maps.luma[k][n] = en->slot[en->lmap[i]].tm_luma[k]; maps.chroma[k][n] = en->slot[en->lmap[i]].tm_chroma[k]; }
        maps.index_of_slot[i] = (int8_t)n++;
        maps.valid_slots |= 1u << i;
      }
      const uint32_t* tw = (const uint32_t*)(dbase + off[12]);  // tile words, then the batch table
      TL("mc", (k_inter_pred_tma<<<std::min(L.n_batches, en->num_sms * en->mc_ctas), MCT_CTA_THREADS, sizeof(MctShared), st>>>(
                   dp, maps, (const b200_pu*)(dbase + off[0]), (const b200_weight_entry*)(dbase + off[1]), tw, tw + n_tiles, L.n_batches)));
    } else {
      k_inter_pred<P><<<(n_tiles + 3) / 4, 128, 0, st>>>(dp, refs, (const b200_pu*)(dbase + off[0]), (const b200_weight_entry*)(dbase + off[1]),
                                                           (const uint32_t*)(dbase + off[12]), n_tiles);
    }
    en->launches++;
  }
  if (en->timing) CU(cudaEventRecord(en->ev[2], st));
  if ((L.n_a > 0 || L.n_b > 0) && L.params.stop_after_stage != B200_STAGE_INTER_PRED) {
    ReconArgs ra;
    ra.tus = (const b200_tu*)(dbase + off[2]);
    ra.coeffs = (const b200_coeff*)(dbase + off[5]);
    ra.scaling = L.has_scaling ? dbase + off[11] : nullptr;
    ra.ticket = (unsigned int*)cx.sync_buf;
    ra.poll_ns = en->poll_ns;
    ra.err = en->intra_err;
    ra.err_host = en->intra_err_host;
    ra.spin_limit_ns = en->spin_limit_ns;
    const size_t cw4 = (size_t)((dp.cw + 3) / 4), ch4 = (size_t)((dp.ch + 3) / 4);
    ra.pend[0] = cx.sync_buf + 256;
    ra.pend[1] = ra.pend[0] + (size_t)dp.w4 * dp.h4;
    ra.pend[2] = ra.pend[1] + cw4 * ch4;
    ra.pend_w[0] = dp.w4;
    ra.pend_w[1] = ra.pend_w[2] = (int)cw4;
    ra.mark_list = nullptr;
    ra.n_mark = 0;
    if (L.n_b > 0) CU(cudaMemsetAsync(cx.sync_buf, 0, 256 + (size_t)dp.w4 * dp.h4 + 2 * cw4 * ch4, st));  // ticket + pending flags
    if (L.n_a > 0) {
      ra.list = (const uint32_t*)(dbase + off[3]);
      ra.n_list = L.n_a;
      ra.n_listw = L.n_aw;
      ra.n_list8 = L.n_a8;
      if (L.n_b > 0) {  // k_residual also sets the pending flags of the intra TUs
        ra.mark_list = (const uint32_t*)(dbase + off[4]);
        ra.n_mark = L.n_b;
      }
      const int items = L.n_aw + (L.n_a8 + 3) / 4 + (L.n_a - L.n_aw - L.n_a8 + 31) / 32;
      TL("residual", (k_residual<P><<<std::min((items + RC_WARPS - 1) / RC_WARPS, en->num_sms * 4), RC_THREADS, 0, st>>>(dp, ra)));
      en->launches++;
    }
    ra.trace = nullptr;
    if (L.n_b > 0) {
      unsigned long long* trace_dev = nullptr;
      const char* trace_path = getenv("B200_TRACE_INTRA");  // debug: per-task timing trace of k_intra appended to this file
      if (trace_path && L.n_task > 0) {
        CU(cudaMalloc(&trace_dev, sizeof(unsigned long long) * 4 * (size_t)L.n_task));
        CU(cudaMemsetAsync(trace_dev, 0, sizeof(unsigned long long) * 4 * (size_t)L.n_task, st));
        ra.trace = trace_dev;
      }
      ra.list = (const uint32_t*)(dbase + off[4]);
      ra.n_list = L.n_b;
      if (L.n_a == 0) {
        TL("mark", (k_mark_pending<<<(L.n_b + 255) / 256, 256, 0, st>>>(ra)));
        en->launches++;
      }
      ra.task_start = (const uint32_t*)(dbase + off[13]);
      ra.n_task = L.n_task;
      int grid = (L.n_task + RC_WARPS - 1) / RC_WARPS;
      // an intra picture's DAG is latency-bound (one CTA per SM is as fast) and should leave room for the pictures it overlaps with
      const bool background = L.ref_mask == 0 && en->n_ctx > 1;
      const int cap = background ? (en->intra_i_grid ? en->intra_i_grid : en->num_sms) : en->num_sms * en->intra_ctas;
      if (grid > cap) grid = cap;
      TL("intra", (k_intra<P><<<grid, RC_THREADS, sizeof(IntraSmem<P>), st>>>(dp, ra)));
      en->launches++;
      if (trace_dev) {
        std::vector<unsigned long long> h(4 * (size_t)L.n_task);
        CU(cudaStreamSynchronize(st));
        CU(cudaMemcpy(h.data(), trace_dev, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        cudaFree(trace_dev);
        if (FILE* f = fopen(trace_path, "ab")) {
          const unsigned long long n = (unsigned long long)L.n_task;
          fwrite(&n, sizeof(n), 1, f);
          fwrite(h.data(), sizeof(unsigned long long), h.size(), f);
          fclose(f);
        }
      }
    }
  }
  if (en->timing) CU(cudaEventRecord(en->ev[3], st));
  FilterArgs fa;
  fa.bs_map = dbase + off[8];
  fa.qp_map = (const int8_t*)(dbase + off[9]);
  fa.nofilt_map = dbase + off[10];
  fa.slices = (const b200_slice_info*)(dbase + off[6]);
  fa.ctbs = (const b200_ctb_info*)(dbase + off[7]);
  if (run_deblock) {
    const int nseg = ((dp.w4 + 1) / 2) * dp.h4 > dp.w4 * ((dp.h4 + 1) / 2) ? ((dp.w4 + 1) / 2) * dp.h4 : dp.w4 * ((dp.h4 + 1) / 2);
    dim3 grid((nseg + 127) / 128, dp.chroma ? 2 : 1);
    TL("deblock_v", (k_deblock<P, true><<<grid, 128, 0, st>>>(dp, fa)));
    TL("deblock_h", (k_deblock<P, false><<<grid, 128, 0, st>>>(dp, fa)));
    en->launches += 2;
  }
  if (en->timing) CU(cudaEventRecord(en->ev[4], st));
  if (run_sao) {
    uint16_t* avail = (uint16_t*)(cx.sync_buf + sync_sao_offset(L.params));
    fa.sao_avail = avail;
    const bool sao8 = sizeof(P) == 1 && dp.log2ctb >= 5;
    if (!sao8) {  // k_sao8 derives the neighbour masks itself
      TL("sao_prep", (k_sao_prep<<<(2 * dp.wctb * dp.hctb + 127) / 128, 128, 0, st>>>(dp, fa, avail)));
      en->launches++;
    }
    dim3 grid((dp.w / 8 + 127) / 128, dp.h, dp.chroma ? 3 : 1);
    if (sao8) {  // byte-parallel kernel: a warp per CTB part (kernels_filter.cuh)
      Sao8Layout lay;
      lay.n_ctb = dp.wctb * dp.hctb;
      const int S = 1 << dp.log2ctb, rows_l = (32 >> (dp.log2ctb - 4)) * SAO8_R, rows_c = (32 >> (dp.log2ctb - 5)) * SAO8_R;
      lay.ipl = (S + rows_l - 1) / rows_l;
      lay.ipc = dp.chroma ? (S / 2 + rows_c - 1) / rows_c : 0;
      const int items = lay.n_ctb * (lay.ipl + 2 * lay.ipc);
      TL("sao", (k_sao8<<<(items + SAO8_WARPS - 1) / SAO8_WARPS, SAO8_WARPS * 32, 0, st>>>(dp, fa, lay)));
    } else {
      TL("sao", (k_sao<P><<<grid, 128, 0, st>>>(dp, fa)));
    }
    en->launches++;
  }
  if (en->timing) CU(cudaEventRecord(en->ev[5], st));
  CU(cudaGetLastError());
  return B200_OK;
}

// Validates the records, groups TUs by CTB, cuts PUs into MC tiles and packs everything into `hb`
// (which must hold L->total bytes; call with hb == nullptr first to size it).
// Section order in the staging buffer / device arena: the raw record arrays first (their offsets depend only on the
// counts, so copying them can start before the work lists exist), then the lists the planner builds.
//   0 pus, 1 weights, 2 tus, 5 coeffs, 6 slices, 7 ctbs, 8 bs_map, 9 qp_map, 10 nofilt_map, 11 scaling |
//   3 list_a (non-intra TU indices by k_residual class), 4 list_b (intra TU indices by task), 12 MC units / tiles, 13 task_start
static const int k_raw_sections[10] = {0, 1, 2, 5, 6, 7, 8, 9, 10, 11};
static const int k_list_sections[4] = {3, 4, 12, 13};

static int plan_begin(b200_engine* en, const b200_picture* pic, PicLayout* L, size_t* cap_total)
{
  const b200_pic_params& p = pic->params;
  int rc = check_params(p);
  if (rc) return rc;
  if ((pic->n_pu && !pic->pus) || (pic->n_tu && !pic->tus) || (pic->n_coeff && !pic->coeffs) || !pic->slices || !pic->ctbs || !pic->qp_map ||
      !pic->nofilt_map || pic->n_slices == 0)
    return set_err(B200_ERR_INVALID, "missing record arrays");
  if (pic->n_pu >= (1u << 20)) return set_err(B200_ERR_INVALID, "too many PUs");
  const int S = 1 << p.log2_ctb_size;
  const int wctb = (p.width + S - 1) / S, hctb = (p.height + S - 1) / S, n_ctb = wctb * hctb;
  const int w4 = (p.width + 3) / 4, h4 = (p.height + 3) / 4, w8 = (p.width + 7) / 8, h8 = (p.height + 7) / 8;
  L->params = p;
  L->n_tu = pic->n_tu;
  L->has_scaling = pic->scaling_factors != nullptr;
  L->run_deblock = !(p.flags & B200_PIC_SKIP_DEBLOCK) && pic->bs_map && (p.stop_after_stage == B200_STAGE_ALL || p.stop_after_stage == B200_STAGE_DEBLOCK);
  L->run_sao = (p.flags & B200_PIC_SAO_ENABLED) && !(p.flags & B200_PIC_SKIP_SAO) && p.stop_after_stage == B200_STAGE_ALL;

  for (int i = 0; i < n_ctb; i++)
    if (pic->ctbs[i].slice_idx >= pic->n_slices) return set_err(B200_ERR_INVALID, "CTB %d slice index", i);
  size_t sz[14] = {};
  sz[0] = sizeof(b200_pu) * pic->n_pu;
  sz[1] = sizeof(b200_weight_entry) * pic->n_weights;
  sz[2] = sizeof(b200_tu) * pic->n_tu;
  sz[5] = sizeof(b200_coeff) * pic->n_coeff;
  sz[6] = sizeof(b200_slice_info) * pic->n_slices;
  sz[7] = sizeof(b200_ctb_info) * (size_t)n_ctb;
  sz[8] = L->run_deblock ? (size_t)w4 * h4 : 0;
  sz[9] = (size_t)w8 * h8;
  sz[10] = (size_t)w8 * h8;
  sz[11] = L->has_scaling ? B200_SCALING_FACTOR_BYTES : 0;
  size_t total = 0;
  for (int i : k_raw_sections) { L->off[i] = total; total += align_up(sz[i], 256); }
  L->raw_total = total;
  L->direct = (p.flags & B200_PIC_RECORDS_PINNED) != 0;
  const void* src[14] = {pic->pus, pic->weights, pic->tus, nullptr, nullptr, pic->coeffs, pic->slices, pic->ctbs, pic->bs_map, pic->qp_map, pic->nofilt_map,
                         pic->scaling_factors, nullptr, nullptr};
  for (int i : k_raw_sections) { L->raw_src[i] = src[i]; L->raw_sz[i] = sz[i]; }
  // upper bound of the lists: every TU in one list, one task per TU; MC units cannot outnumber 4x8 blocks unless PUs overlap
  L->unit_cap = ((size_t)w4 * h4 / 2 + 64 + 8 * MCT_MAX_TILES) * 3 / 2 + 64;  // + the padding of the class-pure batches + the batch table
  *cap_total = total + 3 * align_up(sizeof(uint32_t) * ((size_t)pic->n_tu + 1), 256) + align_up(sizeof(uint32_t) * L->unit_cap, 256) + 256;
  return B200_OK;
}

// PU validation + MC work list for the PU range [i0, i1) into the part's own tile list (parts run on pool threads;
// plan_pus_merge sorts them into class-pure batches)
static int plan_pus_part(b200_engine* en, const b200_picture* pic, int part, uint32_t i0, uint32_t i1)
{
  const b200_pic_params& p = pic->params;
  std::vector<uint32_t>& tiles = en->pu_tiles[part];
  // at most 16 tiles (64x64 PU) per record: written through a raw pointer, trimmed at the end (no per-tile capacity check)
  tiles.resize((size_t)(i1 - i0) * 16);
  uint32_t* out = tiles.data();
  uint32_t ref_mask = 0;
  size_t count[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const bool wide = p.bit_depth_luma > 8;  // same rule as the launch_picture<P> dispatch
  const unsigned pw = p.width, ph = p.height;
  const uint32_t n_weights = pic->n_weights;
  const b200_pu* pus = pic->pus;
  for (uint32_t i = i0; i < i1; i++) {
    const b200_pu& pu = pus[i];
    const unsigned w = pu.w, h = pu.h;
    if (w - 1u > 63u || h - 1u > 63u || ((w | h | pu.x | pu.y) & 3u) || pu.x + w > pw || pu.y + h > ph)
      return set_err(B200_ERR_INVALID, "PU %u out of range", i);
    if ((pu.flags & B200_PU_WEIGHTED) && pu.wt_idx >= n_weights) return set_err(B200_ERR_INVALID, "PU %u weight index", i);
    if (pu.ref_slot[0] >= B200_MAX_SLOTS || pu.ref_slot[1] >= B200_MAX_SLOTS) return set_err(B200_ERR_INVALID, "PU %u reference slot", i);
    const unsigned l0 = pu.flags & B200_PU_PRED_L0, l1 = pu.flags & B200_PU_PRED_L1;
    if (!(l0 | l1)) continue;
    if (l0 && pu.ref_slot[0] >= 0) ref_mask |= 1u << pu.ref_slot[0];
    if (l1 && pu.ref_slot[1] >= 0) ref_mask |= 1u << pu.ref_slot[1];
    if (wide) {  // 16-bit path: <= 16x16 tiles, one warp each (kernels_mc.cuh)
      for (unsigned ty = 0; ty * MC_TILE < h; ty++)
        for (unsigned tx = 0; tx * MC_TILE < w; tx++) *out++ = i | (tx << 20) | (ty << 22);
    } else {     // 8-bit path: <= 16x16 tiles with their class (kernels_mct.cuh), sorted into class-pure batches by the merge
      const unsigned bi = (l0 && l1) ? MCT_CLASS_BI : 0;
      for (unsigned ty = 0; ty * 16 < h; ty++) {
        const unsigned tall = (h - 16 * ty > 8) ? MCT_CLASS_TALL : 0;
        for (unsigned tx = 0; tx * 16 < w; tx++) {
          const unsigned cls = bi | tall | ((w - 16 * tx > 8) ? MCT_CLASS_WIDE : 0);
          *out++ = MCT_TILE_WORD(i, tx, ty, cls);
          count[cls]++;
        }
      }
    }
  }
  tiles.resize((size_t)(out - tiles.data()));
  for (int c = 0; c < 8; c++) en->pu_count[part][c] = count[c];
  en->pu_ref_mask[part] = ref_mask;
  return B200_OK;
}

// Concatenates the parts; 8-bit: counting sort by class, every class padded to whole batches (MCT_CLASS_TILES tiles of one class,
// padding = MCT_INVALID), the batch table (first tile index | class) behind the tile words in the same section.
static int plan_pus_merge(b200_engine* en, const b200_picture* pic, PicLayout* L)
{
  const bool wide = pic->params.bit_depth_luma > 8;
  std::vector<uint32_t>& tiles = en->tiles;
  L->n_batches = 0;
  for (int part = 0; part < PLAN_PU_PARTS; part++) L->ref_mask |= en->pu_ref_mask[part];
  size_t n_words;
  if (wide) {
    tiles.clear();
    for (int part = 0; part < PLAN_PU_PARTS; part++) tiles.insert(tiles.end(), en->pu_tiles[part].begin(), en->pu_tiles[part].end());
    n_words = tiles.size();
  } else {
    size_t count[8] = {}, start[8], total = 0, nb = 0;
    for (int part = 0; part < PLAN_PU_PARTS; part++)
      for (int c = 0; c < 8; c++) count[c] += en->pu_count[part][c];
    for (int c = 0; c < 8; c++) {
      const size_t per = MCT_CLASS_TILES(c), batches = (count[c] + per - 1) / per;
      start[c] = total;
      total += batches * per;
      nb += batches;
    }
    tiles.assign(total + nb, MCT_INVALID);
    size_t bi = total;
    for (int c = 0; c < 8; c++)
      for (size_t f = start[c]; f < start[c] + (count[c] + MCT_CLASS_TILES(c) - 1) / MCT_CLASS_TILES(c) * MCT_CLASS_TILES(c); f += MCT_CLASS_TILES(c))
        tiles[bi++] = MCT_BATCH_WORD(f, c);
    for (int part = 0; part < PLAN_PU_PARTS; part++)
      for (uint32_t t : en->pu_tiles[part]) tiles[start[(t >> 24) & 7]++] = t;
    n_words = total;
    L->n_batches = (int)nb;
  }
  if (tiles.size() > L->unit_cap) return set_err(B200_ERR_INVALID, "PUs overlap (more MC units than the picture has 4x8 blocks)");
  L->n_tiles = (int)n_words;  // tile words; en->tiles also holds the n_batches batch words behind them
  return B200_OK;
}

// TU validation + the k_residual work classes for the TU range [i0, i1) into the part's own lists (two parts run on pool
// threads; plan_and_pack concatenates them).  Classes: warp per TU (16x16, 32x32, PCM) | quarter-warp per 8x8 | lane per 4x4.
#define PLAN_TU_PARTS PLAN_INTRA_PARTS  // validation and the intra task formation share one pass over a range of TUs
// One TU record against the picture; B200_OK or the error (message set).  `dims`: plane sizes per cIdx (0 when the plane does not exist).
struct TuDims { int pw[3], ph[3]; };
static inline TuDims tu_dims(const b200_pic_params& p)
{
  TuDims d;
  d.pw[0] = p.width; d.ph[0] = p.height;
  d.pw[1] = d.pw[2] = p.chroma_format_idc ? p.width / 2 : 0;
  d.ph[1] = d.ph[2] = p.chroma_format_idc ? p.height / 2 : 0;
  return d;
}
static inline int tu_check(const TuDims& d, const b200_picture* pic, uint32_t i, const b200_tu& tu)
{
  const unsigned l2 = tu.log2_size, c = tu.cidx;
  if (l2 - 2u > 3u || c > 2u) return set_err(B200_ERR_INVALID, "TU %u out of range", i);
  const int nT = 1 << l2, pw = d.pw[c], ph = d.ph[c];
  if (tu.x + nT > pw || tu.y + nT > ph || ((tu.x | tu.y) & (nT - 1))) return set_err(B200_ERR_INVALID, "TU %u out of range", i);  // nT >= 4: also the 4-sample grid
  if ((size_t)tu.coeff_off + tu.n_coeff > pic->n_coeff || tu.n_coeff > nT * nT) return set_err(B200_ERR_INVALID, "TU %u coefficient range", i);
  if ((tu.flags & B200_TU_PCM) && tu.n_coeff != nT * nT) return set_err(B200_ERR_INVALID, "PCM TU %u sample count", i);
  if (tu.flags & B200_TU_INTRA) {
    if (tu.intra_mode > 34) return set_err(B200_ERR_INVALID, "TU %u intra mode", i);
    // avail bits must name samples inside the picture (k_intra reads the border and the pending flags at those positions)
    const int half = nT >> 1;  // groups of 4 samples per side
    const uint32_t gm = half >= 32 ? 0xffffffffu : (1u << half) - 1u;
    const uint32_t left = (uint32_t)tu.avail & 0xffffu, top = (uint32_t)(tu.avail >> B200_AVAIL_TOP_BIT0) & 0xffffu;
    const bool corner = (tu.avail >> B200_AVAIL_CORNER_BIT) & 1;
    const int rows_below = (ph - tu.y) >> 2, cols_right = (pw - tu.x) >> 2;  // groups that still lie inside the plane
    const uint32_t lm = rows_below >= 16 ? 0xffffu : (1u << rows_below) - 1u, tm = cols_right >= 16 ? 0xffffu : (1u << cols_right) - 1u;
    if ((left & ~gm) || (top & ~gm) || (tu.avail >> (B200_AVAIL_TOP_BIT0 + 16)) || (left && tu.x == 0) || (top && tu.y == 0) ||
        (corner && (tu.x == 0 || tu.y == 0)) || (left & ~lm) || (top & ~tm))
      return set_err(B200_ERR_INVALID, "TU %u intra availability names samples outside the picture", i);
  }
  return B200_OK;
}

// TU validation, the k_residual classes of the non-intra TUs and the intra work list, in one pass over the TU records.  Intra tasks: the TUs of one plane inside one aligned 16x16-luma / 8x8-chroma region (contiguous per plane in
// decode order); a TU at least as large as the region is a task of its own.  Tasks are ranked in a topological order: DAG level,
// ties in decode order (plan_intra_levels).  The TU list is cut at CTB boundaries into PLAN_INTRA_PARTS ranges (a region never
// crosses a CTB, so no task spans two ranges) and the phases A, C, E run per range on the pool threads:
//   A  per range: intra TUs, their (range-local) task ids                               B  serial: task offsets of the ranges, rank of every task
//   C  per range: TUs per task                                                          D  serial: prefix sum -> task_start
//   E  per range: list_b (TU indices grouped by task in rank order)

static inline uint32_t plan_ctb_of(const b200_pic_params& p, const b200_tu& tu)
{
  const int sh = (tu.cidx && tu.cidx <= 2) ? 1 : 0;
  return (uint32_t)(((uint32_t)tu.x << sh) >> p.log2_ctb_size) | ((uint32_t)(((uint32_t)tu.y << sh) >> p.log2_ctb_size) << 16);
}

static void plan_intra_ranges(b200_engine* en, const b200_picture* pic)
{
  const b200_pic_params& p = pic->params;
  uint32_t prev = 0;
  for (int k = 0; k < PLAN_INTRA_PARTS; k++) {
    uint32_t end = (k == PLAN_INTRA_PARTS - 1) ? pic->n_tu : (uint32_t)((uint64_t)pic->n_tu * (k + 1) / PLAN_INTRA_PARTS);
    if (end < prev) end = prev;
    // move the cut forward to the next CTB change (all TUs of a CTB are contiguous in decode order)
    while (end > 0 && end < pic->n_tu && plan_ctb_of(p, pic->tus[end]) == plan_ctb_of(p, pic->tus[end - 1])) end++;
    en->ipart[k].i0 = prev;
    en->ipart[k].i1 = end;
    prev = end;
  }
}

// One task per plane and region in every picture: merging the planes of a region into one task (fewer tasks, but three dependent
// L2 round trips each) was measured slower, also in pictures with inter prediction (DESIGN.md §4).
static int plan_intra_A(b200_engine* en, const b200_picture* pic, int k)
{
  const b200_pic_params& p = pic->params;
  IntraPart& ip = en->ipart[k];
  std::vector<uint32_t>&la = en->part_a[k][0], &la8 = en->part_a[k][1], &la4 = en->part_a[k][2];  // non-intra TUs with a residual, by k_residual class
  la.clear();
  la8.clear();
  la4.clear();
  ip.intra_idx.clear();
  ip.task_of.clear();
  ip.task_cell.clear();
  const TuDims dims = tu_dims(p);
  long long cur_key[3] = {-1, -1, -1};
  uint32_t cur_task[3] = {0, 0, 0};
  for (uint32_t i = ip.i0; i < ip.i1; i++) {
    const b200_tu& tu = pic->tus[i];
    if (const int rc = tu_check(dims, pic, i, tu)) return rc;
    if (!(tu.flags & B200_TU_INTRA)) {
      if (tu.flags & (B200_TU_CBF | B200_TU_PCM)) {
        if ((tu.flags & B200_TU_PCM) || tu.log2_size > 3) la.push_back(i);
        else if (tu.log2_size == 3) la8.push_back(i);
        else la4.push_back(i);
      }
      continue;
    }
    const int c = tu.cidx, sh = c ? 1 : 0, G = RC_REGION >> sh, nT = 1 << tu.log2_size;
    ip.intra_idx.push_back(i);
    const long long key = (nT >= G) ? -2 - (long long)i : (((long long)(tu.y >> (RC_LG_REGION - sh))) << 20) | (tu.x >> (RC_LG_REGION - sh));
    if (key != cur_key[c]) {
      cur_key[c] = key;
      // what plan_intra_levels needs of the task, kept here so that pass reads no TU record
      const uint32_t R = std::max(1u, ((1u << tu.log2_size) << sh) >> RC_LG_REGION);
      ip.task_cell.push_back((((uint32_t)tu.x << sh) >> RC_LG_REGION) | ((((uint32_t)tu.y << sh) >> RC_LG_REGION) << 12) | (R << 24) | ((uint32_t)c << 28));
      cur_task[c] = (uint32_t)ip.task_cell.size() - 1;
    }
    ip.task_of.push_back(cur_task[c]);
  }
  return B200_OK;
}

static void plan_intra_B(b200_engine* en, uint32_t* n_task, uint32_t* n_intra)
{
  uint32_t nt = 0, ni = 0;
  for (int k = 0; k < PLAN_INTRA_PARTS; k++) {
    en->ipart[k].task_base = nt;
    nt += (uint32_t)en->ipart[k].task_cell.size();
    ni += (uint32_t)en->ipart[k].intra_idx.size();
  }
  *n_task = nt;
  *n_intra = ni;
  en->task_order.resize(nt);
  en->task_start.assign((size_t)nt + 1, 0);
  en->list_b.resize(ni);
}

// Ticket order by DAG LEVEL.  A level is assigned per task in ONE pass over the tasks in decode order through a map per plane
// "region cell (16x16 luma) -> highest level of a task covering it":
//   level(task) = 1 + max over the cells its TUs may read (the column left of it from one cell above to 2x its height below —
//   corner, left and bottom-left neighbours — and the row above it to 2x its width — top and top-right), cells not written yet
//   (decoded later, or not intra) count 0.
// That is a superset of the true dependencies (availability bits), which is all a valid layering needs: every neighbour a task
// waits for has a lower level.  Tasks of one level are independent, so with tickets sorted by level the lowest unfinished
// tickets are exactly the ready tasks: the persistent warps of k_intra hold ready work instead of spinning on tasks far down
// the picture.  (A CTB anti-diagonal order is topological too, but of the ~500 consecutive tickets the warps hold only the
// first task of every CTB chain is ready.)
static void plan_intra_levels(b200_engine* en, const b200_picture* pic, PicLayout* L, uint32_t n_task)
{
  const b200_pic_params& p = pic->params;
  const int cw = (p.width + RC_REGION - 1) >> RC_LG_REGION, ch = (p.height + RC_REGION - 1) >> RC_LG_REGION;
  for (int c = 0; c < 3; c++) en->cell_level[c].assign((size_t)cw * ch, 0);
  std::vector<uint32_t>& level = en->task_level;
  level.resize(n_task);
  uint32_t max_level = 0;
  for (int k = 0; k < PLAN_INTRA_PARTS; k++) {
    const IntraPart& ip = en->ipart[k];
    for (size_t t = 0; t < ip.task_cell.size(); t++) {
      const uint32_t tc = ip.task_cell[t];
      const int cx = (int)(tc & 0xfff), cy = (int)((tc >> 12) & 0xfff);
      const int R = (int)((tc >> 24) & 0xf);  // cells per side: 1 (region task) or the large TU's size
      uint32_t* map = en->cell_level[tc >> 28].data();
      uint32_t lvl = 0;
      if (cx > 0)
        for (int y = std::max(cy - 1, 0); y < std::min(cy + 2 * R, ch); y++) lvl = std::max(lvl, map[(size_t)y * cw + cx - 1]);
      if (cy > 0)
        for (int x = cx; x < std::min(cx + 2 * R, cw); x++) lvl = std::max(lvl, map[(size_t)(cy - 1) * cw + x]);
      lvl++;
      level[ip.task_base + t] = lvl;
      if (lvl > max_level) max_level = lvl;
      for (int y = cy; y < std::min(cy + R, ch); y++)
        for (int x = cx; x < std::min(cx + R, cw); x++) {
          uint32_t& m = map[(size_t)y * cw + x];
          if (lvl > m) m = lvl;  // several tasks may cover a cell (large chroma TUs)
        }
    }
  }
  // rank = position in (level, decode order): counting sort over the levels
  std::vector<uint32_t>& off = en->level_off;
  off.assign((size_t)max_level + 2, 0);
  for (uint32_t t = 0; t < n_task; t++) off[level[t] + 1]++;
  uint32_t width = 0;
  for (size_t l = 1; l < off.size(); l++) {
    if (off[l] > width) width = off[l];
    off[l] += off[l - 1];
  }
  uint32_t* order = en->task_order.data();
  for (uint32_t t = 0; t < n_task; t++) order[t] = off[level[t]]++;
  L->intra_levels = (int)max_level;
  L->intra_width = (int)width;
}

static void plan_intra_C(b200_engine* en, int k)
{
  const IntraPart& ip = en->ipart[k];
  const uint32_t* order = en->task_order.data() + ip.task_base;
  uint32_t* ts = en->task_start.data();
  for (size_t j = 0; j < ip.task_of.size(); j++) ts[order[ip.task_of[j]] + 1]++;  // a task belongs to exactly one range: no two threads touch one entry
}

static void plan_intra_E(b200_engine* en, int k)
{
  IntraPart& ip = en->ipart[k];
  const uint32_t* order = en->task_order.data() + ip.task_base;
  const uint32_t* ts = en->task_start.data();
  ip.fill.resize(ip.task_cell.size());
  for (size_t t = 0; t < ip.task_cell.size(); t++) ip.fill[t] = ts[order[t]];
  uint32_t* lb = en->list_b.data();
  for (size_t j = 0; j < ip.intra_idx.size(); j++) lb[ip.fill[ip.task_of[j]]++] = ip.intra_idx[j];
}

// Runs `f(k)` for k = 0..n-1 on the pool (or inline without one) and waits.
template <typename F>
static void plan_parallel(b200_engine* en, int n, F f)
{
  for (int k = 0; k < n; k++) en->prun([=] { f(k); });
  en->pwait();
}

// The serial glue of the intra planner after phase A has run for every range (also used by plan_and_pack, where phase A runs
// next to the other planning work).
static void plan_intra_finish(b200_engine* en, const b200_picture* pic, PicLayout* L)
{
  uint32_t n_task = 0, n_intra = 0;
  plan_intra_B(en, &n_task, &n_intra);
  L->intra_levels = L->intra_width = 0;
  if (n_task) plan_intra_levels(en, pic, L, n_task);
  plan_parallel(en, PLAN_INTRA_PARTS, [=](int k) { plan_intra_C(en, k); });
  uint32_t* ts = en->task_start.data();
  for (uint32_t t = 0; t < n_task; t++) ts[t + 1] += ts[t];
  plan_parallel(en, PLAN_INTRA_PARTS, [=](int k) { plan_intra_E(en, k); });
  L->n_task = (int)n_task;
  L->n_b = (int)n_intra;
}

static void plan_finish(PicLayout* L)
{
  size_t sz[14] = {};
  sz[3] = sizeof(uint32_t) * (size_t)L->n_a;
  sz[4] = sizeof(uint32_t) * (size_t)L->n_b;
  sz[12] = sizeof(uint32_t) * (size_t)(L->n_tiles + L->n_batches);
  sz[13] = L->n_task ? sizeof(uint32_t) * (size_t)(L->n_task + 1) : 0;
  size_t total = L->raw_total;
  for (int i : k_list_sections) { L->off[i] = total; total += align_up(sz[i], 256); }
  L->total = total ? total : 256;
}

// part 0..2: the raw record arrays in three roughly equal shares (pool threads)
static void pack_raw(const b200_picture* pic, const PicLayout& L, uint8_t* hb, int part)
{
  const b200_pic_params& p = pic->params;
  const size_t* off = L.off;
  const int S = 1 << p.log2_ctb_size;
  const int wctb = (p.width + S - 1) / S, hctb = (p.height + S - 1) / S, n_ctb = wctb * hctb;
  const int w4 = (p.width + 3) / 4, h4 = (p.height + 3) / 4, w8 = (p.width + 7) / 8, h8 = (p.height + 7) / 8;
  if (part == 0) {
    if (pic->n_coeff) memcpy(hb + off[5], pic->coeffs, sizeof(b200_coeff) * pic->n_coeff);
  } else if (part == 1) {
    if (pic->n_tu) memcpy(hb + off[2], pic->tus, sizeof(b200_tu) * pic->n_tu);
    memcpy(hb + off[6], pic->slices, sizeof(b200_slice_info) * pic->n_slices);
    memcpy(hb + off[7], pic->ctbs, sizeof(b200_ctb_info) * (size_t)n_ctb);
  } else {
    if (pic->n_pu) memcpy(hb + off[0], pic->pus, sizeof(b200_pu) * pic->n_pu);
    if (pic->n_weights) memcpy(hb + off[1], pic->weights, sizeof(b200_weight_entry) * pic->n_weights);
    if (L.run_deblock) memcpy(hb + off[8], pic->bs_map, (size_t)w4 * h4);
    memcpy(hb + off[9], pic->qp_map, (size_t)w8 * h8);
    memcpy(hb + off[10], pic->nofilt_map, (size_t)w8 * h8);
    if (L.has_scaling) memcpy(hb + off[11], pic->scaling_factors, B200_SCALING_FACTOR_BYTES);
  }
}

static void pack_lists(b200_engine* en, const PicLayout& L, uint8_t* hb)
{
  const size_t* off = L.off;
  if (L.n_a) memcpy(hb + off[3], en->list_a.data(), sizeof(uint32_t) * (size_t)L.n_a);
  if (L.n_b) memcpy(hb + off[4], en->list_b.data(), sizeof(uint32_t) * (size_t)L.n_b);
  if (L.n_task) memcpy(hb + off[13], en->task_start.data(), sizeof(uint32_t) * (size_t)(L.n_task + 1));
  if (L.n_tiles) memcpy(hb + off[12], en->tiles.data(), sizeof(uint32_t) * (size_t)(L.n_tiles + L.n_batches));
}

// cap_hint = the largest staging capacity any set of the engine has needed: a set that has to grow goes straight to it, so that
// every set is reallocated at most once after the first large (intra) picture instead of whenever such a picture happens to land
// on it (page-locking tens of MB and cudaFree both stall the other threads' CUDA calls).

static int ensure_staging(StagingSet& ss, size_t total)
{
  if (ss.in_flight) { CU(cudaEventSynchronize(ss.done)); ss.in_flight = false; }
  std::atomic<size_t> local{0};
  std::atomic<size_t>& cap_hint = ss.cap_hint ? *ss.cap_hint : local;
  size_t hint = cap_hint.load(std::memory_order_relaxed);
  const size_t want = align_up(total + total / 2, 1 << 20);
  while (want > hint && !cap_hint.compare_exchange_weak(hint, want, std::memory_order_relaxed)) {}
  if (ss.cap < total) {
    if (ss.host) cudaFreeHost(ss.host);
    if (ss.dev) cudaFree(ss.dev);
    ss.host = nullptr; ss.dev = nullptr;
    ss.cap = std::max(want, cap_hint.load(std::memory_order_relaxed));
    CU(cudaMallocHost(&ss.host, ss.cap));
    CU(cudaMalloc(&ss.dev, ss.cap));
  }
  return B200_OK;
}

// list_a = class by class (warp | 8x8 | 4x4), the validation parts in order
static void merge_list_a(b200_engine* en, PicLayout* L)
{
  std::vector<uint32_t>& la = en->list_a;
  la.clear();
  for (int cls = 0; cls < 3; cls++) {
    for (int part = 0; part < PLAN_TU_PARTS; part++) la.insert(la.end(), en->part_a[part][cls].begin(), en->part_a[part][cls].end());
    if (cls == 0) L->n_aw = (int)la.size();
    if (cls == 1) L->n_a8 = (int)la.size() - L->n_aw;
  }
  L->n_a = (int)la.size();
}

// Host side of one picture: validate, build the work lists, fill the pinned staging buffer.  The raw record arrays are
// copied by pool threads and the PUs are planned on a pool thread while this thread plans the TUs.
static int plan_and_pack(b200_engine* en, const b200_picture* pic, PicLayout* L, StagingSet& ss, double* t_plan_pack)
{
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t0 = now();
  size_t cap = 0;
  int rc = plan_begin(en, pic, L, &cap);
  if (rc) return rc;
  rc = ensure_staging(ss, cap);
  if (rc) return rc;
  const double t1 = now();
  uint8_t* hb = ss.host;
  en->use_helper = en->helper && pic->n_tu > 200000;  // shadow engines: see b200_engine::helper
  int rc_pu[PLAN_PU_PARTS] = {}, rc_tv[PLAN_TU_PARTS] = {};
  std::string err_pu[PLAN_PU_PARTS], err_tv[PLAN_TU_PARTS];
  plan_intra_ranges(en, pic);
  for (int k = 0; k < PLAN_INTRA_PARTS; k++)  // the longest items first: TU validation + residual classes + intra tasks of one range
    en->prun([&, k] {
      rc_tv[k] = plan_intra_A(en, pic, k);
      if (rc_tv[k]) err_tv[k] = g_err;  // the worker's thread-local message
    });
  for (int part = 0; part < PLAN_PU_PARTS; part++) {
    const uint32_t i0 = (uint32_t)((uint64_t)pic->n_pu * part / PLAN_PU_PARTS), i1 = (uint32_t)((uint64_t)pic->n_pu * (part + 1) / PLAN_PU_PARTS);
    en->prun([&, part, i0, i1] {
      rc_pu[part] = plan_pus_part(en, pic, part, i0, i1);
      if (rc_pu[part]) err_pu[part] = g_err;  // the worker's thread-local message
    });
  }
  if (!L->direct)
    for (int part = 0; part < 3; part++) en->prun([=] { pack_raw(pic, *L, hb, part); });
  en->pwait();
  for (int part = 0; part < PLAN_TU_PARTS; part++)
    if (rc_tv[part]) return set_err(rc_tv[part], "%s", err_tv[part].c_str());
  for (int part = 0; part < PLAN_PU_PARTS; part++)
    if (rc_pu[part]) return set_err(rc_pu[part], "%s", err_pu[part].c_str());
  plan_intra_finish(en, pic, L);
  merge_list_a(en, L);
  rc = plan_pus_merge(en, pic, L);
  if (rc) return rc;
  plan_finish(L);
  pack_lists(en, *L, hb);
  if (t_plan_pack) { t_plan_pack[0] = t1 - t0; t_plan_pack[1] = now() - t1; }
  return B200_OK;
}

extern "C" int b200_plan_picture_host(const b200_picture* pic, uint32_t counts[8], uint32_t* mc_units, size_t cap_units, uint32_t* list_a, size_t cap_a,
                                      uint32_t* list_b, size_t cap_b, uint32_t* task_start, size_t cap_tasks)
{
  if (!pic || !counts) return set_err(B200_ERR_INVALID, "null argument");
  b200_engine* en = new (std::nothrow) b200_engine();  // no CUDA call is made on this path
  if (!en) return set_err(B200_ERR_NOMEM, "out of memory");
  PicLayout L;
  size_t cap = 0;
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const bool prof = getenv("B200_HOST_PROF") != nullptr;
  double t[5] = {now(), 0, 0, 0, 0};
  int rc = plan_begin(en, pic, &L, &cap);
  t[1] = now();
  for (int part = 0; part < PLAN_PU_PARTS && !rc; part++)
    rc = plan_pus_part(en, pic, part, (uint32_t)((uint64_t)pic->n_pu * part / PLAN_PU_PARTS), (uint32_t)((uint64_t)pic->n_pu * (part + 1) / PLAN_PU_PARTS));
  if (!rc) rc = plan_pus_merge(en, pic, &L);
  t[2] = now();
  t[3] = now();
  if (!rc) {
    plan_intra_ranges(en, pic);
    for (int k = 0; k < PLAN_INTRA_PARTS && !rc; k++) rc = plan_intra_A(en, pic, k);
    if (!rc) plan_intra_finish(en, pic, &L);
  }
  t[4] = now();
  if (prof) {
    double u[4];
    u[0] = now();
    for (int part = 0; part < PLAN_PU_PARTS && !rc; part++) en->pu_ref_mask[part] = 0;
    if (!rc) rc = plan_pus_merge(en, pic, &L);
    u[1] = now();
    if (!rc) plan_intra_finish(en, pic, &L);
    u[2] = now();
    merge_list_a(en, &L);
    u[3] = now();
    fprintf(stderr, "[b200] intra DAG: %d tasks in %d levels, widest level %d tasks\n", L.n_task, L.intra_levels, L.intra_width);
    fprintf(stderr, "[b200] plan (one thread) ms: begin %.3f  PUs %.3f  (-) %.3f  TU validate + intra tasks %.3f | serial tail: PU merge %.3f  intra finish %.3f  list_a merge %.3f\n",
            1e3 * (t[1] - t[0]), 1e3 * (t[2] - t[1]), 1e3 * (t[3] - t[2]), 1e3 * (t[4] - t[3]), 1e3 * (u[1] - u[0]), 1e3 * (u[2] - u[1]), 1e3 * (u[3] - u[2]));
  }
  if (!rc) {
    merge_list_a(en, &L);
    plan_finish(&L);
    counts[0] = (uint32_t)L.n_tiles; counts[1] = (uint32_t)L.n_a; counts[2] = (uint32_t)L.n_aw; counts[3] = (uint32_t)L.n_a8;
    counts[4] = (uint32_t)L.n_b; counts[5] = (uint32_t)L.n_task; counts[6] = L.ref_mask; counts[7] = 0;
    auto copy = [](uint32_t* dst, size_t cap_, const std::vector<uint32_t>& v, size_t n) {
      if (dst) memcpy(dst, v.data(), sizeof(uint32_t) * std::min(cap_, n));
    };
    copy(mc_units, cap_units, en->tiles, (size_t)L.n_tiles);
    copy(list_a, cap_a, en->list_a, (size_t)L.n_a);
    copy(list_b, cap_b, en->list_b, (size_t)L.n_b);
    copy(task_start, cap_tasks, en->task_start, L.n_task ? (size_t)L.n_task + 1 : 0);
  }
  delete en;
  return rc;
}

// Is every access to physical surface `ph` issued on a stream other than `k` complete?  (Same-stream accesses are ordered anyway.)
static bool phys_idle(b200_engine* en, int ph, int k)
{
  SlotSync& ss = en->ssync[ph];
  if (ss.writer >= 0 && ss.writer != k) {
    if (cudaEventQuery(ss.written) != cudaSuccess) return false;
    ss.writer = -1;
  }
  for (int c = 0; c < B200_MAX_CTX; c++)
    if (c != k && ss.read_pending[c]) {
      if (cudaEventQuery(ss.read[c]) != cudaSuccess) return false;
      ss.read_pending[c] = false;
    }
  cudaGetLastError();  // cudaErrorNotReady is not sticky, but leave nothing behind
  return true;
}

static bool same_geometry(const Surface& s, const b200_pic_params& p)
{
  return s.plane[0] && s.w == p.width && s.h == p.height && s.chroma == p.chroma_format_idc &&
         bytes_per_sample(s.bd_y) == bytes_per_sample(p.bit_depth_luma) && bytes_per_sample(s.bd_c) == bytes_per_sample(p.bit_depth_chroma);
}

// The physical surface a picture issued on stream `k` writes for the name `d` (see b200_engine::slot).
static int phys_for_write(b200_engine* en, int d, int k, const b200_pic_params& p)
{
  const int cur = en->lmap[d];
  if (cur >= 0 && (en->n_ctx <= 1 || en->timing || phys_idle(en, cur, k))) return cur;
  int best = -1, empty = -1, other = -1;
  for (int ph = 0; ph < B200_MAX_PHYS && best < 0; ph++) {
    if (en->owner[ph] >= 0) continue;
    const Surface& s = en->slot[ph];
    if (!s.plane[0]) { if (empty < 0) empty = ph; continue; }
    if (!phys_idle(en, ph, k)) continue;
    if (same_geometry(s, p)) best = ph;
    else if (other < 0) other = ph;
  }
  if (best < 0) best = empty >= 0 ? empty : other;  // a new surface, or an idle one of another format (surface_ensure reallocates it)
  if (best < 0) return cur;                         // pool exhausted: write in place behind the readers (order_before waits)
  if (cur >= 0) {
    en->owner[cur] = -1;
    en->n_renamed++;
  }
  en->lmap[d] = best;
  en->owner[best] = d;
  en->last_owner[best] = d;
  return best;
}

// Cross-stream ordering for a picture issued on context `k` (SlotSync, per physical surface): wait for the writers of its
// reference surfaces and for every earlier reader / writer of its destination surface that ran on another stream (none when the
// destination was renamed to an idle surface).
static int order_before(b200_engine* en, int k, const PicLayout& L, int dst_phys)
{
  cudaStream_t st = en->ctx[k].stream;
  const int d = L.params.dst_slot;
  for (int r = 0; r < B200_MAX_SLOTS; r++) {
    if (!((L.ref_mask >> r) & 1) || r == d || en->lmap[r] < 0) continue;
    SlotSync& ss = en->ssync[en->lmap[r]];
    if (ss.writer >= 0 && ss.writer != k) CU(cudaStreamWaitEvent(st, ss.written, 0));
  }
  SlotSync& sd = en->ssync[dst_phys];
  if (sd.writer >= 0 && sd.writer != k) CU(cudaStreamWaitEvent(st, sd.written, 0));
  for (int c = 0; c < B200_MAX_CTX; c++)
    if (c != k && sd.read_pending[c]) CU(cudaStreamWaitEvent(st, sd.read[c], 0));
  return B200_OK;
}

static int order_after(b200_engine* en, int k, const PicLayout& L, int dst_phys)
{
  cudaStream_t st = en->ctx[k].stream;
  const int d = L.params.dst_slot;
  if (en->n_ctx > 1) {
    for (int r = 0; r < B200_MAX_SLOTS; r++) {
      if (!((L.ref_mask >> r) & 1) || r == d || en->lmap[r] < 0) continue;
      SlotSync& sr = en->ssync[en->lmap[r]];
      CU(cudaEventRecord(sr.read[k], st));
      sr.read_pending[k] = true;
    }
  }
  SlotSync& sd = en->ssync[dst_phys];
  CU(cudaEventRecord(sd.written, st));
  sd.writer = k;
  for (auto& rp : sd.read_pending) rp = false;  // this picture waited for them; later pictures wait for this one
  return B200_OK;
}

// Everything after the records are in device memory at `dbase`.  `upload_from`: pinned source to copy first (or null).
static int run_layout(b200_engine* en, int k, const PicLayout& L, uint8_t* dbase, const uint8_t* upload_from)
{
  PipeCtx& cx = en->ctx[k];
  const b200_pic_params& p = L.params;
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const bool prof = en->host_prof && en->async && en->host_skip <= 0;
  double tseg[5] = {prof ? now() : 0.0, 0, 0, 0, 0};
  // references resolve against the names as they are BEFORE this picture takes its destination name
  RefTable refs;
  memset(&refs, 0, sizeof(refs));
  for (int i = 0; i < B200_MAX_SLOTS; i++) {
    if (i == p.dst_slot || en->lmap[i] < 0) continue;
    const Surface& s = en->slot[en->lmap[i]];
    if (s.valid && s.w == p.width && s.h == p.height && s.chroma == p.chroma_format_idc && s.bd_y == p.bit_depth_luma && s.bd_c == p.bit_depth_chroma)
      for (int c = 0; c < 3; c++) refs.plane[i][c] = s.plane[c];
  }
  {
    // Format change (new SPS): drain, then drop every surface that carries no name — surfaces of another format cannot be reused
    // as they are, and converting them one rename at a time (free + allocate, each a device-wide synchronisation) was measured
    // to leave the second format at 75 % of its speed for a long time.
    const uint64_t geom = (uint64_t)p.width | ((uint64_t)p.height << 16) | ((uint64_t)p.chroma_format_idc << 32) |
                          ((uint64_t)bytes_per_sample(p.bit_depth_luma) << 34) | ((uint64_t)bytes_per_sample(p.bit_depth_chroma) << 36);
    if (en->pool_geom && en->pool_geom != geom) {
      for (int c = 0; c < B200_MAX_CTX; c++) CU(cudaStreamSynchronize(en->ctx[c].stream));
      for (int ph = 0; ph < B200_MAX_PHYS; ph++)
        if (en->owner[ph] < 0 && en->slot[ph].plane[0] && !same_geometry(en->slot[ph], p)) surface_free(en->slot[ph]);
    }
    en->pool_geom = geom;
  }
  int dst_phys = phys_for_write(en, p.dst_slot, k, p);
  if (dst_phys < 0) {  // first use of the name with every surface taken: cannot happen (B200_MAX_PHYS > B200_MAX_SLOTS), but stay safe
    return set_err(B200_ERR_NOMEM, "no free picture surface");
  }
  Surface& dst = en->slot[dst_phys];
  int rc = surface_ensure(dst, p, cx.stream);
  if (rc) return rc;
  Surface* cur = &dst;
  if (L.run_sao) {
    rc = surface_ensure(cx.scratch, p, cx.stream);
    if (rc) return rc;
    cur = &cx.scratch;
  }
  {
    const size_t n_ctb = (size_t)((p.width + (1 << p.log2_ctb_size) - 1) >> p.log2_ctb_size) * ((p.height + (1 << p.log2_ctb_size) - 1) >> p.log2_ctb_size);
    const size_t need = sync_sao_offset(p) + 2 * n_ctb * sizeof(uint16_t);
    if (cx.sync_cap < need) {
      if (cx.sync_buf) { CU(cudaStreamSynchronize(cx.stream)); cudaFree(cx.sync_buf); }
      cx.sync_buf = nullptr;
      CU(cudaMalloc(&cx.sync_buf, need));
      cx.sync_cap = need;
    }
  }
  cudaStream_t st = cx.stream;
  en->ev = en->timing ? &en->tev[(size_t)(en->tcount % TIMING_RING) * 7] : nullptr;
  if (en->timing) CU(cudaEventRecord(en->ev[0], st));
  if (upload_from && L.direct) {  // raw record arrays straight from the caller's page-locked memory, the planner's lists from the staging buffer
    for (int i : k_raw_sections)
      if (L.raw_sz[i]) CU(cudaMemcpyAsync(dbase + L.off[i], L.raw_src[i], L.raw_sz[i], cudaMemcpyHostToDevice, st));
    if (L.total > L.raw_total) CU(cudaMemcpyAsync(dbase + L.raw_total, upload_from + L.raw_total, L.total - L.raw_total, cudaMemcpyHostToDevice, st));
  } else if (upload_from) {
    CU(cudaMemcpyAsync(dbase, upload_from, L.total, cudaMemcpyHostToDevice, st));  // records first: overlaps the waits below
  }
  if (prof) tseg[1] = now();
  rc = order_before(en, k, L, dst_phys);
  if (rc) return rc;
  if (prof) tseg[2] = now();
  const DevPic dp = make_devpic(p, *cur, dst);
  if (p.bit_depth_luma > 8) rc = launch_picture<uint16_t>(en, cx, L, dp, refs, dbase);
  else rc = launch_picture<uint8_t>(en, cx, L, dp, refs, dbase);
  if (rc) return rc;
  if (prof) tseg[3] = now();
  if (en->tl_path) tl_begin(en, st, "extend", L.params.poc, k);
  launch_extend_borders(dst, st);  // the finished picture may be referenced: replicate its edges into the border
  if (en->tl_path) tl_end(en, st);
  en->launches++;
  CU(cudaGetLastError());
  if (en->timing) { CU(cudaEventRecord(en->ev[6], st)); en->tcount++; }
  rc = order_after(en, k, L, dst_phys);
  if (rc) return rc;
  dst.valid = true;
  if (prof) {
    tseg[4] = now();
    for (int i = 0; i < 4; i++) en->async_s[4 + i] += tseg[i + 1] - tseg[i];
  }
  return B200_OK;
}

// Per-stage timing needs the stages of consecutive pictures not to overlap: one stream while it is on.
// Pictures that read no reference (intra pictures) go to a stream of their own: nothing queued in front of them, so the
// long intra DAG of the next intra period's I picture runs in the background of the current period's P/B pictures.
//
// The other pictures are placed by DEPENDENCY DEPTH (depth = 1 + the largest depth among the pictures in the slots it reads): a
// stream is a FIFO, so a picture queued behind an unrelated picture that still waits for ITS references is held up for nothing
// (round-robin puts the next GOP's key picture behind the current GOP's leaf B pictures: 16 picture times per 4 GOPs instead
// of 7).  A picture goes to the stream whose last picture has the largest depth still below its own (that picture finishes
// before this one could start anyway); if there is none, to the stream whose last picture is the shallowest.
static uint32_t ref_mask_of(const b200_picture* pic)
{
  uint32_t m = 0;
  for (uint32_t i = 0; i < pic->n_pu; i++) {
    const b200_pu& pu = pic->pus[i];
    if ((pu.flags & B200_PU_PRED_L0) && pu.ref_slot[0] >= 0 && pu.ref_slot[0] < B200_MAX_SLOTS) m |= 1u << pu.ref_slot[0];
    if ((pu.flags & B200_PU_PRED_L1) && pu.ref_slot[1] >= 0 && pu.ref_slot[1] < B200_MAX_SLOTS) m |= 1u << pu.ref_slot[1];
  }
  return m;
}

static int pick_ctx(b200_engine* en, uint32_t ref_mask, int dst_slot)
{
  if (en->timing || en->n_ctx <= 1) return 0;
  long long depth = 1;
  for (int r = 0; r < B200_MAX_SLOTS; r++)
    if ((ref_mask >> r) & 1) depth = std::max(depth, en->slot_depth[r] + 1);
  int k;
  if (ref_mask == 0 && en->n_ctx + en->n_ind <= B200_MAX_CTX) {  // the long intra DAGs of consecutive intra pictures overlap each other too
    // an all-intra stream (several pictures in a row that read no reference) spreads over ALL streams: every picture is a
    // latency-bound DAG on a quarter of the SMs, so many of them fit side by side
    en->ind_run++;
    const int pool = en->ind_run > 2 ? en->n_ctx + en->n_ind : en->n_ind, base = en->ind_run > 2 ? 0 : en->n_ctx;
    k = base + en->next_ind % pool;
    en->next_ind = (en->next_ind + 1) % pool;
    depth = en->key_depth + 1;  // what references it comes after the pictures already queued
  } else {
    int best = -1, shallow = 0;
    for (int c = 0; c < en->n_ctx; c++) {
      if (en->tail_depth[c] < depth && (best < 0 || en->tail_depth[c] > en->tail_depth[best])) best = c;
      if (en->tail_depth[c] < en->tail_depth[shallow]) shallow = c;
    }
    k = best >= 0 ? best : shallow;
  }
  if (ref_mask != 0) en->ind_run = 0;
  en->tail_depth[k] = depth;
  if (dst_slot >= 0 && dst_slot < B200_MAX_SLOTS) en->slot_depth[dst_slot] = depth;
  en->key_depth = std::max(en->key_depth, depth);
  return k;
}

// ---- asynchronous submission ------------------------------------------------------------------------------------------------
// b200_engine_submit_picture spends ~1 ms of host time per 4K picture (validation, work lists, packing), spread over the pool
// threads but with serial joins; a host that produces pictures faster than that (a parser with several slice / WPP threads, a
// cache of recorded pictures, bench.py's e2e leg) is held up by it.  The asynchronous path plans WHOLE pictures in parallel: the
// caller only queues the picture; N planner threads (each with private scratch: a "shadow" engine without CUDA state) validate /
// plan / pack one picture each into its staging set; ONE sequencer thread takes the queue in submission order, waits for the
// picture's plan, and issues the copies and kernels exactly as the synchronous path does — so stream placement, DPB ordering and
// results are identical.  Reads of finished pictures (b200_engine_read_slot_async) are queued behind the picture they follow.
struct AsyncCmd {
  int kind = 0;  // 0 picture, 1 read slot
  b200_picture pic{};
  PicLayout L;
  StagingSet* ss = nullptr;
  int rc = B200_OK;
  std::string err;
  int state = 0;  // 0 queued, 1 being planned, 2 planned (guarded by AsyncState::m)
  int slot = 0;
  void* planes[3] = {nullptr, nullptr, nullptr};
  size_t strides[3] = {0, 0, 0};
  unsigned long long seq = 0;  // ticket: position in submission order (1, 2, ...)
};
struct AsyncState {
  std::mutex m;
  std::condition_variable cv_plan, cv_seq, cv_space;
  std::deque<AsyncCmd*> q;  // submission order; the front is the next one the sequencer executes
  int n_pictures = 0;       // pictures in q (read-backs do not count towards the depth)
  int depth = 12;           // pictures queued at most (B200_ASYNC_QUEUE; <= B200_ASYNC_DEPTH)
  std::vector<std::thread> planners;
  std::thread sequencer;
  std::vector<b200_engine*> shadows;
  bool stop = false;
  int first_rc = B200_OK;
  std::string first_err;
  unsigned long long enq_seq = 0, done_seq = 0;          // tickets: queued last / issued last
  unsigned long long slot_seq[B200_MAX_SLOTS] = {};      // ticket of the last queued command that writes or reads the slot
};
#define B200_ASYNC_DEPTH 32  // queued PICTURES; < B200_STAGE_SETS: a staging set is never handed out again before its previous picture was launched

static int run_layout(b200_engine* en, int k, const PicLayout& L, uint8_t* dbase, const uint8_t* upload_from);
static int pick_ctx(b200_engine* en, uint32_t ref_mask, int dst_slot);
static int read_slot_async_now(b200_engine* en, int slot, void* const planes[3], const size_t strides[3]);

// Cores this process may use: the affinity mask, clamped by the cgroup v2 CPU quota.
static int host_cores()
{
  int n = (int)std::thread::hardware_concurrency();
  cpu_set_t set;
  if (sched_getaffinity(0, sizeof(set), &set) == 0) n = CPU_COUNT(&set);
  if (FILE* f = fopen("/sys/fs/cgroup/cpu.max", "r")) {
    char quota[32] = "";
    long period = 0;
    if (fscanf(f, "%31s %ld", quota, &period) == 2 && strcmp(quota, "max") != 0 && period > 0) n = std::min(n, std::max(1, (int)((atol(quota) + period - 1) / period)));
    fclose(f);
  }
  return std::max(1, n);
}

static inline double prof_now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

static void async_planner(b200_engine* en, b200_engine* shadow)
{
  AsyncState* as = en->async;
  cudaSetDevice(en->device);
  for (;;) {
    AsyncCmd* cmd = nullptr;
    {
      std::unique_lock<std::mutex> lk(as->m);
      for (;;) {
        if (as->stop) return;
        for (AsyncCmd* c : as->q)
          if (c->kind == 0 && c->state == 0) { cmd = c; break; }
        if (cmd) break;
        as->cv_plan.wait(lk);
      }
      cmd->state = 1;
    }
    const double tp0 = en->host_prof ? prof_now() : 0.0;
    const int rc = plan_and_pack(shadow, &cmd->pic, &cmd->L, *cmd->ss, nullptr);
    const double tp1 = en->host_prof ? prof_now() : 0.0;
    {
      std::lock_guard<std::mutex> lk(as->m);
      if (en->host_skip <= 0) en->async_s[0] += tp1 - tp0;
      cmd->rc = rc;
      if (rc) cmd->err = g_err;
      cmd->state = 2;
    }
    as->cv_seq.notify_all();
  }
}

static void async_sequencer(b200_engine* en)
{
  AsyncState* as = en->async;
  cudaSetDevice(en->device);
  for (;;) {
    AsyncCmd* cmd = nullptr;
    double ts[3] = {0, 0, 0};
    {
      std::unique_lock<std::mutex> lk(as->m);
      as->cv_seq.wait(lk, [&] { return as->stop || !as->q.empty(); });  // an empty queue is idle time, not waiting for a plan
      if (as->stop) return;
      if (en->host_prof) ts[0] = prof_now();
      as->cv_seq.wait(lk, [&] { return as->stop || (!as->q.empty() && (as->q.front()->kind != 0 || as->q.front()->state == 2)); });
      if (as->stop) return;
      cmd = as->q.front();
    }
    if (en->host_prof) ts[1] = prof_now();
    int rc = cmd->rc;
    {
      std::lock_guard<std::mutex> issue(en->issue_m);
      if (cmd->kind == 0) {
        if (!rc) {
          const int k = pick_ctx(en, cmd->L.ref_mask, cmd->L.params.dst_slot);
          rc = run_layout(en, k, cmd->L, cmd->ss->dev, cmd->ss->host);
          if (!rc) {
            cudaEventRecord(cmd->ss->done, en->ctx[k].stream);
            cmd->ss->in_flight = true;
          }
        }
      } else {
        rc = read_slot_async_now(en, cmd->slot, cmd->planes, cmd->strides);
      }
    }
    if (en->host_prof && en->host_skip > 0) {
      if (cmd->kind == 0) en->host_skip--;  // B200_HOST_PROF_SKIP: warm-up pictures (first-use allocations) stay out of the profile
    } else if (en->host_prof) {
      ts[2] = prof_now();
      en->async_s[1] += ts[1] - ts[0];
      en->async_s[cmd->kind == 0 ? 2 : 3] += ts[2] - ts[1];
      if (cmd->kind == 0) en->async_n++;
    }
    {
      std::lock_guard<std::mutex> lk(as->m);
      if (rc && !as->first_rc) { as->first_rc = rc; as->first_err = cmd->err.empty() ? std::string(g_err) : cmd->err; }
      as->q.pop_front();
      if (cmd->kind == 0) as->n_pictures--;
      as->done_seq = cmd->seq;
    }
    delete cmd;
    as->cv_space.notify_all();
    as->cv_seq.notify_all();
  }
}

static int async_start(b200_engine* en)
{
  if (en->async) return B200_OK;
  AsyncState* as = new (std::nothrow) AsyncState();
  if (!as) return set_err(B200_ERR_NOMEM, "out of memory");
  en->async = as;
  // one planner takes ~4 ms of one core per 4K picture: the cores this process may use (affinity mask and cgroup quota: exceeding
  // the quota gets the whole process throttled) minus four for the caller, the sequencer and the CUDA driver's threads, at most 16
  // (B200_ASYNC_THREADS overrides)
  int n = std::max(2, std::min(16, host_cores() - 4));
  if (const char* e = getenv("B200_ASYNC_THREADS")) n = std::max(1, std::min(32, atoi(e)));
  as->depth = std::min(B200_ASYNC_DEPTH, n + 8);
  if (const char* e = getenv("B200_ASYNC_QUEUE")) as->depth = std::max(1, std::min(B200_ASYNC_DEPTH, atoi(e)));
  try {  // thread creation may throw (resource limits): no exception leaves the C ABI
    as->sequencer = std::thread(async_sequencer, en);
    for (int i = 0; i < n; i++) {
      b200_engine* sh = new b200_engine();  // no CUDA state: only the planner's scratch
      sh->device = en->device;
      sh->helper = &en->pool;
      as->shadows.push_back(sh);
      as->planners.emplace_back(async_planner, en, sh);
    }
  } catch (const std::exception& ex) {
    if (as->planners.empty() || !as->sequencer.joinable()) {  // nothing usable: tear down what exists
      async_stop(en);
      return set_err(B200_ERR_NOMEM, "asynchronous submission: cannot start threads (%s)", ex.what());
    }
    // fewer planners than asked for still work
    as->depth = std::min(as->depth, (int)as->planners.size() + 8);
  }
  return B200_OK;
}

// Blocks until every queued command has been issued to the GPU; returns (and clears) the first error of a queued command.
static int async_flush(b200_engine* en)
{
  AsyncState* as = en->async;
  if (!as) return B200_OK;
  std::unique_lock<std::mutex> lk(as->m);
  as->cv_space.wait(lk, [&] { return as->q.empty(); });
  const int rc = as->first_rc;
  if (rc) set_err(rc, "%s", as->first_err.c_str());
  as->first_rc = B200_OK;
  as->first_err.clear();
  return rc;
}

// Blocks until every command up to `ticket` has been issued (its records are no longer read by the host side).
static int async_wait_ticket(b200_engine* en, unsigned long long ticket)
{
  AsyncState* as = en->async;
  if (!as) return B200_OK;
  std::unique_lock<std::mutex> lk(as->m);
  if (ticket > as->enq_seq) ticket = as->enq_seq;  // a ticket that was never handed out: everything queued so far
  as->cv_space.wait(lk, [&] { return as->done_seq >= ticket; });
  const int rc = as->first_rc;
  if (rc) set_err(rc, "%s", as->first_err.c_str());
  as->first_rc = B200_OK;
  as->first_err.clear();
  return rc;
}

static void async_stop(b200_engine* en)
{
  AsyncState* as = en->async;
  if (!as) return;
  async_flush(en);
  {
    std::lock_guard<std::mutex> lk(as->m);
    as->stop = true;
  }
  as->cv_plan.notify_all();
  as->cv_seq.notify_all();
  for (auto& t : as->planners) t.join();
  if (as->sequencer.joinable()) as->sequencer.join();
  for (b200_engine* sh : as->shadows) delete sh;
  delete as;
  en->async = nullptr;
}

static int async_enqueue(b200_engine* en, AsyncCmd* cmd)
{
  AsyncState* as = en->async;
  {
    std::unique_lock<std::mutex> lk(as->m);
    as->cv_space.wait(lk, [&] { return as->n_pictures < as->depth && as->q.size() < 4 * B200_ASYNC_DEPTH; });
    as->q.push_back(cmd);
    if (cmd->kind == 0) as->n_pictures++;
    cmd->seq = ++as->enq_seq;
    const int slot = cmd->kind == 0 ? (int)cmd->pic.params.dst_slot : cmd->slot;
    if (slot >= 0 && slot < B200_MAX_SLOTS) as->slot_seq[slot] = cmd->seq;
  }
  if (cmd->kind == 0) as->cv_plan.notify_one();
  as->cv_seq.notify_all();
  return B200_OK;
}

extern "C" int b200_engine_submit_picture_async(b200_engine* en, const b200_picture* pic)
{
  if (!en || !pic) return set_err(B200_ERR_INVALID, "null argument");
  CU(cudaSetDevice(en->device));
  int rc = async_start(en);
  if (rc) return rc;
  AsyncCmd* cmd = new (std::nothrow) AsyncCmd();
  if (!cmd) return set_err(B200_ERR_NOMEM, "out of memory");
  cmd->kind = 0;
  cmd->pic = *pic;  // the record ARRAYS must stay valid until b200_engine_flush / _sync returns
  cmd->ss = &en->stage_pool[en->next_stage++ % B200_STAGE_SETS];
  return async_enqueue(en, cmd);
}

extern "C" unsigned long long b200_engine_last_ticket(b200_engine* en)
{
  if (!en || !en->async) return 0;
  std::lock_guard<std::mutex> lk(en->async->m);
  return en->async->enq_seq;
}

extern "C" int b200_engine_wait_ticket(b200_engine* en, unsigned long long ticket)
{
  if (!en) return set_err(B200_ERR_INVALID, "null engine");
  return async_wait_ticket(en, ticket);
}

extern "C" int b200_engine_flush(b200_engine* en)
{
  if (!en) return set_err(B200_ERR_INVALID, "null engine");
  return async_flush(en);
}

extern "C" int b200_engine_submit_picture(b200_engine* en, const b200_picture* pic)
{
  if (!en || !pic) return set_err(B200_ERR_INVALID, "null argument");
  CU(cudaSetDevice(en->device));
  {
    const int frc = async_flush(en);  // keep submission order with pictures queued asynchronously
    if (frc) return frc;
  }
  PicLayout L;
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const int k = pick_ctx(en, ref_mask_of(pic), pic->params.dst_slot);
  PipeCtx& cx = en->ctx[k];
  StagingSet& ss = en->stage_pool[en->next_stage++ % B200_STAGE_SETS];
  double tp[2] = {0, 0};
  int rc = plan_and_pack(en, pic, &L, ss, tp);
  if (rc) return rc;
  const double t3 = now();
  rc = run_layout(en, k, L, ss.dev, ss.host);
  if (rc) return rc;
  CU(cudaEventRecord(ss.done, cx.stream));
  ss.in_flight = true;
  if (en->host_skip > 0) en->host_skip--;  // B200_HOST_PROF_SKIP: leave the warm-up (first-use allocations) out of the profile
  else { en->host_s[0] += tp[0]; en->host_s[1] += tp[1]; en->host_s[3] += now() - t3; en->host_n++; }
  return B200_OK;
}

extern "C" int b200_engine_prepare_picture(b200_engine* en, const b200_picture* pic, b200_prepared** out)
{
  if (!en || !pic || !out) return set_err(B200_ERR_INVALID, "null argument");
  CU(cudaSetDevice(en->device));
  { const int frc = async_flush(en); if (frc) return frc; }
  b200_prepared* pp = new (std::nothrow) b200_prepared();
  if (!pp) return set_err(B200_ERR_NOMEM, "out of memory");
  PipeCtx& cx = en->ctx[0];
  StagingSet& ss = en->stage_pool[en->next_stage++ % B200_STAGE_SETS];
  b200_picture staged = *pic;
  staged.params.flags &= ~B200_PIC_RECORDS_PINNED;  // a prepared picture keeps its own device copy of everything
  int rc = plan_and_pack(en, &staged, &pp->L, ss, nullptr);
  if (rc) { delete pp; return rc; }
  cudaError_t e = cudaMalloc(&pp->dev, pp->L.total);
  if (e == cudaSuccess) e = cudaMemcpyAsync(pp->dev, ss.host, pp->L.total, cudaMemcpyHostToDevice, cx.stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(cx.stream);
  if (e != cudaSuccess) {
    if (pp->dev) cudaFree(pp->dev);
    delete pp;
    return set_err(B200_ERR_CUDA, "prepare: %s", cudaGetErrorString(e));
  }
  *out = pp;
  return B200_OK;
}

extern "C" int b200_engine_run_prepared(b200_engine* en, b200_prepared* pp)
{
  if (!en || !pp) return set_err(B200_ERR_INVALID, "null argument");
  CU(cudaSetDevice(en->device));
  { const int frc = async_flush(en); if (frc) return frc; }
  return run_layout(en, pick_ctx(en, pp->L.ref_mask, pp->L.params.dst_slot), pp->L, pp->dev, nullptr);
}

extern "C" void b200_engine_free_prepared(b200_engine* en, b200_prepared* pp)
{
  if (!en || !pp) return;
  cudaSetDevice(en->device);
  async_flush(en);
  sync_all(en);
  if (pp->dev) cudaFree(pp->dev);
  delete pp;
}

extern "C" int b200_engine_sync(b200_engine* en)
{
  if (!en) return set_err(B200_ERR_INVALID, "null engine");
  CU(cudaSetDevice(en->device));
  { const int frc = async_flush(en); if (frc) return frc; }
  return sync_all(en);
}

template <typename P>
__global__ void k_fill(uint8_t* base, int pitch, int w, int h, int value)
{
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x < w && y < h) row_ptr<P>(base, pitch, y)[x] = (P)value;
}

extern "C" int b200_engine_fill_slot(b200_engine* en, int slot, const b200_pic_params* p, int vy, int vc)
{
  if (!en || !p || slot < 0 || slot >= B200_MAX_SLOTS) return set_err(B200_ERR_INVALID, "bad argument");
  int rc = check_params(*p);
  if (rc) return rc;
  CU(cudaSetDevice(en->device));
  { const int frc = async_flush(en); if (frc) return frc; }
  rc = sync_all(en);  // utility call: quiesce, then write on stream 0
  if (rc) return rc;
  cudaStream_t st = en->ctx[0].stream;
  const int ph = phys_for_write(en, slot, 0, *p);  // everything is idle after sync_all: the name keeps its surface, or gets its first one
  if (ph < 0) return set_err(B200_ERR_NOMEM, "no free picture surface");
  Surface& s = en->slot[ph];
  rc = surface_ensure(s, *p, st);
  if (rc) return rc;
  for (int c = 0; c < (s.chroma ? 3 : 1); c++) {
    const int w = c ? s.cw : s.w, h = c ? s.ch : s.h;
    dim3 grid((w + 255) / 256, h);
    if (p->bit_depth_luma > 8) k_fill<uint16_t><<<grid, 256, 0, st>>>(s.plane[c], s.pitch[c], w, h, c ? vc : vy);
    else k_fill<uint8_t><<<grid, 256, 0, st>>>(s.plane[c], s.pitch[c], w, h, c ? vc : vy);
    en->launches++;
  }
  launch_extend_borders(s, st);
  en->launches++;
  CU(cudaGetLastError());
  CU(cudaEventRecord(en->ssync[ph].written, st));
  en->ssync[ph].writer = 0;
  s.valid = true;
  return B200_OK;
}

extern "C" int b200_engine_upload_slot(b200_engine* en, int slot, const b200_pic_params* p, const void* const planes[3], const size_t strides[3])
{
  if (!en || !p || !planes || !strides || slot < 0 || slot >= B200_MAX_SLOTS) return set_err(B200_ERR_INVALID, "bad argument");
  int rc = check_params(*p);
  if (rc) return rc;
  CU(cudaSetDevice(en->device));
  { const int frc = async_flush(en); if (frc) return frc; }
  rc = sync_all(en);  // utility call: quiesce, then write on stream 0
  if (rc) return rc;
  cudaStream_t st = en->ctx[0].stream;
  const int ph = phys_for_write(en, slot, 0, *p);  // everything is idle after sync_all: the name keeps its surface, or gets its first one
  if (ph < 0) return set_err(B200_ERR_NOMEM, "no free picture surface");
  Surface& s = en->slot[ph];
  rc = surface_ensure(s, *p, st);
  if (rc) return rc;
  for (int c = 0; c < (s.chroma ? 3 : 1); c++) {
    const int w = c ? s.cw : s.w, h = c ? s.ch : s.h, bps = bytes_per_sample(c ? s.bd_c : s.bd_y);
    if (!planes[c]) return set_err(B200_ERR_INVALID, "plane %d missing", c);
    CU(cudaMemcpy2DAsync(s.plane[c], s.pitch[c], planes[c], strides[c], (size_t)w * bps, h, cudaMemcpyHostToDevice, st));
  }
  launch_extend_borders(s, st);
  en->launches++;
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(st));  // the source may be pageable / reused by the caller
  s.valid = true;
  return B200_OK;
}

extern "C" int b200_engine_read_slot_async(b200_engine* en, int slot, void* const planes[3], const size_t strides[3])
{
  if (!en || !planes || !strides || slot < 0 || slot >= B200_MAX_SLOTS) return set_err(B200_ERR_INVALID, "bad argument");
  if (en->async) {  // pictures are queued: the read takes its place behind them (the picture it reads may not be launched yet)
    AsyncCmd* cmd = new (std::nothrow) AsyncCmd();
    if (!cmd) return set_err(B200_ERR_NOMEM, "out of memory");
    cmd->kind = 1;
    cmd->slot = slot;
    for (int c = 0; c < 3; c++) { cmd->planes[c] = planes[c]; cmd->strides[c] = strides[c]; }
    return async_enqueue(en, cmd);
  }
  return read_slot_async_now(en, slot, planes, strides);
}

static int read_slot_async_now(b200_engine* en, int slot, void* const planes[3], const size_t strides[3])
{
  const int ph = en->lmap[slot];
  if (ph < 0 || !en->slot[ph].valid) return set_err(B200_ERR_INVALID, "slot %d holds no picture", slot);
  const Surface& s = en->slot[ph];
  CU(cudaSetDevice(en->device));
  // on the stream of the slot's last writer: ordered after it without an event, and a read other streams must respect
  SlotSync& ss = en->ssync[ph];
  const int k = ss.writer >= 0 ? ss.writer : 0;
  cudaStream_t st = en->ctx[k].stream;
  for (int c = 0; c < (s.chroma ? 3 : 1); c++) {
    if (!planes[c]) continue;
    const int w = c ? s.cw : s.w, h = c ? s.ch : s.h, bps = bytes_per_sample(c ? s.bd_c : s.bd_y);
    CU(cudaMemcpy2DAsync(planes[c], strides[c], s.plane[c], s.pitch[c], (size_t)w * bps, h, cudaMemcpyDeviceToHost, st));
  }
  CU(cudaEventRecord(ss.read[k], st));
  ss.read_pending[k] = true;
  return B200_OK;
}

extern "C" int b200_engine_read_slot(b200_engine* en, int slot, void* const planes[3], const size_t strides[3])
{
  int rc = b200_engine_read_slot_async(en, slot, planes, strides);
  if (rc) return rc;
  rc = async_flush(en);
  if (rc) return rc;
  const int ph = en->lmap[slot];
  const int k = ph >= 0 && en->ssync[ph].writer >= 0 ? en->ssync[ph].writer : 0;
  CU(cudaStreamSynchronize(en->ctx[k].stream));
  return check_intra_err(en);
}

extern "C" int b200_engine_wait_slot(b200_engine* en, int slot)
{
  if (!en || slot < 0 || slot >= B200_MAX_SLOTS) return set_err(B200_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(en->device));
  if (en->async) {  // not a flush: only the commands that touch this slot (later pictures may still be with the planners)
    unsigned long long t;
    {
      std::lock_guard<std::mutex> lk(en->async->m);
      t = en->async->slot_seq[slot];
    }
    const int frc = async_wait_ticket(en, t);
    if (frc) return frc;
  }
  std::vector<cudaEvent_t> evs;
  {
    std::lock_guard<std::mutex> issue(en->issue_m);  // the sequencer may be issuing later pictures
    for (int ph = 0; ph < B200_MAX_PHYS; ph++) {
      // the surface that carries the name, and surfaces that carried it before a later picture took the name elsewhere: a
      // read-back requested from them may still be in flight
      const bool current = en->lmap[slot] == ph;
      if (!current && !(en->owner[ph] < 0 && en->last_owner[ph] == slot)) continue;
      SlotSync& ss = en->ssync[ph];
      if (current && ss.writer >= 0) evs.push_back(ss.written);
      for (int c = 0; c < B200_MAX_CTX; c++)
        if (ss.read_pending[c]) evs.push_back(ss.read[c]);
    }
  }
  for (cudaEvent_t e : evs) CU(cudaEventSynchronize(e));
  return check_intra_err(en);
}

extern "C" void* b200_host_alloc(size_t bytes)
{
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
  return p;
}
extern "C" void b200_host_free(void* p)
{
  if (p) cudaFreeHost(p);
}

extern "C" int b200_engine_slot_device_planes(b200_engine* en, int slot, void* planes[3], size_t strides[3])
{
  if (!en || !planes || !strides || slot < 0 || slot >= B200_MAX_SLOTS) return set_err(B200_ERR_INVALID, "bad argument");
  if (en->lmap[slot] < 0 || !en->slot[en->lmap[slot]].valid) return set_err(B200_ERR_INVALID, "slot %d holds no picture", slot);
  const Surface& s = en->slot[en->lmap[slot]];
  for (int c = 0; c < 3; c++) { planes[c] = s.plane[c]; strides[c] = (size_t)s.pitch[c]; }
  return B200_OK;
}
#include "dsp_table.cuh"
