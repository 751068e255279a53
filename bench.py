#!/usr/bin/env python3
"""bench.py — decoded frames/s of the reconstruction hot path on BASELINE.json's 4K Main random-access config.

A "step" is one intra period of 32 pictures at 3840x2160 8-bit 4:2:0 in decode order (1 I + 3 P + 28 B,
hierarchical-B GOP 8, deblocking + SAO on) replayed from synthetic command records (no HEVC encoder exists
offline, SURVEY §8d).  Lines printed (one JSON object, rank 0):
  value     frames/s with the records already resident in HBM (b200_engine_run_prepared), device-timed
  e2e       frames/s through the C-ABI with HOST buffers: b200_engine_submit_picture (pack + H2D of the records)
            and a D2H read of every finished picture into pinned host memory inside the timed region
  roofline  the dominant kernel (and the MC kernel, the one BASELINE's roofline target names) vs measured HBM peak
  cpu_baseline  the same records replayed on the host cores by the CPU restatement (bounded sample)
--impl reference times the CPU arm alone with all host threads.
N GPUs (torchrun): every rank decodes its own independent stream (BASELINE config 5) - no data-path collective.
"""
import argparse
import ctypes as C
import json
import os

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")  # before CUDA initialises: one hardware queue per engine stream (see capi.py)

import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, BD = 3840, 2160, 8
GOP = [8, 4, 2, 6, 1, 3, 5, 7]  # decode order inside a hierarchical-B GOP (POC offsets)
GOP_REFS = {8: (0, None), 4: (0, 8), 2: (0, 4), 6: (4, 8), 1: (0, 2), 3: (2, 4), 5: (4, 6), 7: (6, 8)}


# DPB slot policy of the synthetic decoder (what dpb.cc's "first unused image" does for libde265, which keeps up to 30
# images, dpb.h:101): 32 slots in three rotating pools — key pictures (POC % 8 == 0) 8 slots, reference B pictures (POC % 8 in
# 2,4,6) 8 slots, non-reference B pictures (odd POC) 16 slots.  A slot is reused only long after its old content stopped being
# referenced or read out, so a new picture never waits for readers of the picture it overwrites (no WAR stalls), and the
# assignment repeats every two intra periods: the workload is 64 prepared pictures, a step alternates between its halves.
KEY_SLOTS, REFB_SLOTS, NONREF_SLOTS = 8, 8, 16
if os.environ.get("B200_TIGHT_DPB"):  # experiment: the smallest DPB the GOP structure allows (7 slots, every slot reused at once): the
    KEY_SLOTS, REFB_SLOTS, NONREF_SLOTS = 2, 3, 2  # WAR / WAW hazards the engine's slot renaming removes (tools/sweep_bench.py)
STEP_VARIANTS = 2


def build_workload(width, height, bd, seed0=1000):
    """Random-access workload (BASELINE configs 3 and 4): 2 x 32 pictures in decode order from 6 generated base pictures (slots
    are patched per use).  Returns (pictures, slot of the key picture the very first GOP references, generation seconds)."""
    from libde265_b200 import synth
    t0 = time.time()
    base = {
        "I": synth.make_picture(width, height, "I", seed=seed0, bit_depth=bd),
        "P": synth.make_picture(width, height, "P", seed=seed0 + 1, bit_depth=bd, ref_slots=(0,)),
    }
    for i in range(4):
        base[f"B{i}"] = synth.make_picture(width, height, "B", seed=seed0 + 2 + i, bit_depth=bd, ref_slots=(0, 1), weighted=(i == 3))
    seq = []
    bcount = 0
    n_key = n_refb = n_nonref = 0
    slot_of = {0: (KEY_SLOTS - 1)}  # POC -> slot; POC 0 = the key picture before the first GOP
    first_key_slot = slot_of[0]
    for g in range(4 * STEP_VARIANTS):  # pocs g*8+1 .. g*8+8, previous key picture at g*8
        for off in GOP:
            poc = g * 8 + off
            if off == 8:
                slot_of[poc] = n_key % KEY_SLOTS
                n_key += 1
            elif off % 2 == 0:
                slot_of[poc] = KEY_SLOTS + n_refb % REFB_SLOTS
                n_refb += 1
            else:
                slot_of[poc] = KEY_SLOTS + REFB_SLOTS + n_nonref % NONREF_SLOTS
                n_nonref += 1
            r0, r1 = GOP_REFS[off]
            ref_a = slot_of[g * 8 + r0]
            ref_b = slot_of[g * 8 + (r1 if r1 is not None else r0)]
            if off == 8:
                kind = "I" if g % 4 == 3 else "P"  # one intra picture per 32
            else:
                kind = f"B{bcount % 4}"
                bcount += 1
            b = base[kind]
            pus = b.pus.copy()
            if len(pus):
                lut = np.array([ref_a, ref_b], np.int8)
                rs = pus["ref_slot"]
                pus["ref_slot"] = np.where(rs >= 0, lut[np.clip(rs, 0, 1)], rs)
            params = type(b.params).from_buffer_copy(b.params)
            params.dst_slot = slot_of[poc]
            params.poc = poc
            seq.append(synth.SynthPicture(params, pus, b.weights, b.tus, b.coeffs, b.slices, b.ctbs, b.bs_map, b.qp_map, b.nofilt_map))
    assert slot_of[32 * STEP_VARIANTS] == first_key_slot, "the slot assignment must repeat after the last variant"
    return seq, first_key_slot, time.time() - t0


_PINNED = {}  # data pointer -> array kept registered for the life of the process


def pin_records(seq, torch):
    """Page-locks the record arrays of the pictures (cudaHostRegister, once per distinct array) and marks the pictures
    B200_PIC_RECORDS_PINNED: the e2e leg's inputs then are pinned host memory the engine uploads from directly (the contract's
    'host->device copy of that step's inputs from pinned host memory').  Returns False (nothing marked) if registration fails."""
    rt = torch.cuda.cudart()
    for p in seq:
        for name in ("pus", "weights", "tus", "coeffs", "slices", "ctbs", "bs_map", "qp_map", "nofilt_map"):
            arr = getattr(p, name)
            if arr is None or arr.size == 0 or arr.ctypes.data in _PINNED:
                continue
            rc = rt.cudaHostRegister(arr.ctypes.data, arr.nbytes, 0)
            if int(rc) != 0:
                return False
            _PINNED[arr.ctypes.data] = arr
    for p in seq:
        p.c.params.flags |= capi_flags().PIC_RECORDS_PINNED
    return True


def unpin_records(seq, torch):
    """Undo pin_records: page-locked memory is a shared resource of the host (later legs and the decoder's own page-locked picture
    planes were measured to slow down with gigabytes of it registered)."""
    rt = torch.cuda.cudart()
    for ptr in list(_PINNED):
        rt.cudaHostUnregister(ptr)
        del _PINNED[ptr]
    for p in seq:
        p.c.params.flags &= ~capi_flags().PIC_RECORDS_PINNED


def capi_flags():
    from libde265_b200 import capi
    return capi


def build_intra_workload(width, height, bd, seed0=3000, n_base=4):
    """All-intra workload (BASELINE config 2): 2 x 32 I pictures from `n_base` generated pictures, destination slots rotating
    over 16 DPB slots.  Intra pictures depend on nothing, so the engine pipelines them over its streams."""
    from libde265_b200 import synth
    t0 = time.time()
    base = [synth.make_picture(width, height, "I", seed=seed0 + i, bit_depth=bd) for i in range(n_base)]
    seq = []
    for i in range(32 * STEP_VARIANTS):
        b = base[i % n_base]
        params = type(b.params).from_buffer_copy(b.params)
        params.dst_slot = i % 16
        params.poc = i
        seq.append(synth.SynthPicture(params, b.pus, b.weights, b.tus, b.coeffs, b.slices, b.ctbs, b.bs_map, b.qp_map, b.nofilt_map))
    return seq, None, time.time() - t0


# The bench configurations: BASELINE.json configs 3 (the headline the metric is quoted on), 2 and 4
CONFIGS = {
    "main_ra_4k": dict(width=3840, height=2160, bd=8, kind="ra", mix=(1, 3, 28),
                       what="3840x2160 8-bit 4:2:0 synthetic command records, hierarchical-B GOP8, intra period 32 (1 I + 3 P + 28 B per step), "
                            "deblock+SAO on, one independent stream per GPU"),
    "main10_4k": dict(width=3840, height=2160, bd=10, kind="ra", mix=(1, 3, 28),
                      what="3840x2160 10-bit 4:2:0 (Main10: 16-bit sample path) synthetic command records, hierarchical-B GOP8, intra period 32 "
                           "(1 I + 3 P + 28 B per step), deblock+SAO on"),
    "intra1080": dict(width=1920, height=1080, bd=8, kind="intra", mix=(32, 0, 0),
                      what="1920x1080 8-bit 4:2:0 synthetic command records, intra-only CTBs (32 I pictures per step, IDCT + intra path), deblock+SAO on"),
}


def algorithmic_bytes(seq, bd):
    """SURVEY §8(d) per-kernel algorithmic bytes, summed over the step's pictures."""
    bps = 2 if bd > 8 else 1
    out = {"inter_pred": 0, "recon": 0, "deblock": 0, "sao": 0}
    for p in seq:
        pic_bytes = (p.params.width * p.params.height * 3 // 2) * bps
        out["inter_pred"] += p.algorithmic_mc_bytes()
        tu = p.tus
        if len(tu):
            px = (1 << (2 * tu["log2_size"].astype(np.int64)))
            intra = (tu["flags"] & 1) != 0
            cbf = (tu["flags"] & 2) != 0
            # residual: 4 B per coefficient + 1 R + 1 W of the touched samples; intra: 1 W per sample + 4nT+1 border reads; + record
            out["recon"] += int(4 * len(p.coeffs) + (2 * px * cbf).sum() * bps + (px * intra).sum() * bps +
                                ((4 * (1 << tu["log2_size"].astype(np.int64)) + 1) * intra).sum() * bps + 24 * len(tu))
        out["deblock"] += 2 * (2 * pic_bytes) + len(p.bs_map) + 2 * len(p.qp_map)
        out["sao"] += 2 * pic_bytes + 24 * len(p.ctbs)
    return out


class ClockSampler:
    def __init__(self, dev):
        self.dev, self.rows, self.proc = dev, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.dev}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [int(r[0]) for r in self.rows if r and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": int(statistics.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons}


METRIC = "decoded frames/sec at 4K Main profile, bit-exact YUV; MC kernel HBM GB/s"  # BASELINE.json


def effective_cores():
    """Host cores this process may really use: the scheduler affinity mask clamped by the cgroup CPU quota (a 1-GPU lease
    on a 128-core node owns a share of it; os.cpu_count() would oversubscribe and inflate every GPU/CPU ratio)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:  # cgroup v2
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
    except (OSError, ValueError):
        try:  # cgroup v1
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except (OSError, ValueError):
            pass
    eff = n if quota is None else max(1, min(n, int(quota + 0.5)))
    return eff, {"affinity": n, "cgroup_quota": None if quota is None else round(quota, 2), "os_cpu_count": os.cpu_count()}


def cpu_replay_worker(args):
    """One host core: generates one picture of the given type and replays it `reps` times through the REFERENCE's own
    reconstruction functions on its SIMD table (oracle/_ref/libref_replay.so, oracle/ref_replay.cc), or — only when oracle/_ref
    was not shipped — through the scalar port.  Returns (type, pictures, seconds, kind) — generation excluded."""
    seed0, width, height, bd, reps, ptype = args
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib  # CPU baseline leg: the only place bench.py touches oracle/
    from libde265_b200 import synth
    kind = "reference" if oracle_lib.ref_replay_lib() is not None else "port"
    orc = oracle_lib.RefReplay(simd=True) if kind == "reference" else oracle_lib.Oracle()
    if ptype == "I":
        pic = synth.make_picture(width, height, "I", seed=seed0, bit_depth=bd, dst_slot=2)
    else:
        pic = synth.make_picture(width, height, ptype, seed=seed0, bit_depth=bd, ref_slots=(0, 1) if ptype == "B" else (0,), dst_slot=2)
        for s in (0, 1):
            orc.upload_slot(s, pic.params, synth.random_planes(width, height, bd, s + 1))
    orc.reconstruct(pic)  # warm-up: page in the surfaces
    t0 = time.time()
    for _ in range(reps):
        orc.reconstruct(pic)
    dt = time.time() - t0
    orc.close()
    return ptype, reps, dt, kind


def cpu_baseline_parallel(width, height, bd, reps, mix=(1, 3, 28), cores=None):
    """The CPU arm: every usable host core busy at once, one independent stream per core (the CPU analogue of one stream per
    GPU, and the most CPU-friendly reading of "all host threads": no synchronisation between cores at all).  Cores replay I, P
    or B pictures; the job rate is `cores` streams of the workload's own picture mix at the measured per-type seconds per
    picture under that full load.  A one-core run first gives the unloaded per-core rate (scaling check of the core count)."""
    import multiprocessing as mp
    info = {}
    if cores is None:
        cores, info = effective_cores()
    nI, nP, nB = mix
    if nP == 0 and nB == 0:
        types = ["I"] * cores
    else:
        types = ["I" if i % 16 == 1 else "P" if i % 8 == 2 else "B" for i in range(cores)] if cores >= 3 else ["B"] * cores
        if cores >= 3 and "I" not in types:
            types[1] = "I"
        if cores >= 3 and "P" not in types:
            types[2] = "P"
    ctx = mp.get_context("spawn")
    with ctx.Pool(1) as pool:  # unloaded single-core rate of the dominant picture type
        solo = pool.map(cpu_replay_worker, [(1002, width, height, bd, max(2, reps // 2), types[0])])[0]
    with ctx.Pool(cores) as pool:
        res = pool.map(cpu_replay_worker, [(1002 + i % 4, width, height, bd, reps, types[i]) for i in range(cores)])
    sec = {}
    for t in ("I", "P", "B"):
        rs = [r for r in res if r[0] == t]
        if rs:
            sec[t] = sum(r[2] for r in rs) / sum(r[1] for r in rs)  # seconds per picture on one core, all cores loaded
    dom = types[0]
    sec.setdefault("B", sec.get("I"))
    sec.setdefault("I", sec["B"])
    sec.setdefault("P", sec["B"])
    step_s = nI * sec["I"] + nP * sec["P"] + nB * sec["B"]
    n = sum(r[1] for r in res)
    kind = res[0][3]
    value = cores * (nI + nP + nB) / step_s
    solo_s = solo[2] / solo[1]
    how = ("the REFERENCE's own reconstruction functions on its SIMD table (generate_inter_prediction_samples, decode_intra_prediction, "
           "scale_coefficients, edge_filtering_*, apply_sample_adaptive_offset_sequential via oracle/_ref/libref_replay.so; "
           "de265_acceleration_AUTO = SSE4.1+AVX2+AVX-512 where present); reconstruction only, no parsing"
           if kind == "reference" else "the CPU restatement oracle/hevc_oracle.c (scalar C, -O3): oracle/_ref not shipped")
    return {"value": round(value, 3), "unit": "frames/s", "cores": cores, "kind": kind, "frames_per_s_per_core": round(value / cores, 3),
            "core_count_source": info,
            "one_core_alone": {"picture_type": dom, "s_per_picture": round(solo_s, 4), "loaded_s_per_picture": round(sec[dom], 4),
                               "parallel_efficiency": round(solo_s / sec[dom], 3)},
            "sample": f"{n} replays of synthetic {width}x{height} {bd}-bit pictures ({reps}/core on {cores} processes: {types.count('I')} I, {types.count('P')} P, "
                      f"{types.count('B')} B cores; {sec['I']:.3f}/{sec['P']:.3f}/{sec['B']:.3f} s per I/P/B picture and core), combined in the workload's mix "
                      f"{nI} I + {nP} P + {nB} B, by {how}"}


# real intra-only streams made with the reference's own encoder (tests/golden/make_intra_streams.py)
REAL_STREAMS = {"1080p_intra": ("intra1080.h265", "1920x1080 intra, 2 pictures"), "4k_intra": ("intra4k.h265", "3840x2160 intra, 1 picture")}


def real_stream_reference(repeats=3, copies=4):
    """Real bitstreams at BASELINE config 2's size and at 4K, the REAL reference: oracle/_ref/libde265_ref.so (SIMD table)
    decoding them through the de265.h API, one thread (the streams have one slice per picture and no WPP)."""
    from libde265_b200 import de265
    lib = os.path.join(ROOT, "oracle", "_ref", "libde265_ref.so")
    if not os.path.exists(lib):
        return {"error": "oracle/_ref/libde265_ref.so not shipped"}
    out = {}
    for key, (fname, what) in REAL_STREAMS.items():
        data = open(os.path.join(ROOT, "tests", "golden", fname), "rb").read() * copies
        best = 0.0
        for _ in range(repeats):
            dec = de265.Decoder(lib)
            t0 = time.time()
            n = dec.decode_stream(data, lambda img: None)
            dt = time.time() - t0
            dec.close()
            best = max(best, n / dt)
        out[key] = {"stream": f"tests/golden/{fname} ({what}) x {copies}", "value": round(best, 2), "unit": "frames/s", "kind": "reference", "cores": 1,
                    "note": "full decode incl. parsing"}
    return out


def real_stream_b200(eng, repeats=3, copies=4):
    """The same streams through the drop-in path, selected the way an application would: DE265_DECODER_PARAM_ACCELERATION_CODE =
    de265_acceleration_B200 on a libde265 built with the binding of INTEGRATION.md (test artefact oracle/_ref/libde265_hooked.so).
    The decoder owns its engine, submits every picture asynchronously and awaits the read-back when the picture is handed out;
    the application fetches pictures one de265_decode call late, so parsing picture N+1 overlaps the GPU work of picture N.  Each
    stream is fed `copies` times back to back (every copy starts with parameter sets + IDR) so that there is something to overlap;
    the reference arm decodes the same bytes."""
    from libde265_b200 import de265
    lib = os.path.join(ROOT, "oracle", "_ref", "libde265_hooked.so")
    if not os.path.exists(lib):
        return {"error": "oracle/_ref/libde265_hooked.so not shipped"}
    out = {}
    for key, (fname, what) in REAL_STREAMS.items():
        data = open(os.path.join(ROOT, "tests", "golden", fname), "rb").read() * copies
        best = 0.0
        for _ in range(repeats):
            dec = de265.Decoder(lib)
            dec.select_b200()
            t0 = time.time()
            n = dec.decode_stream(data, lambda img: None, lag=1)
            dt = time.time() - t0
            dec.close()
            best = max(best, n / dt)
        out[key] = {"stream": f"tests/golden/{fname} ({what}) x {copies}", "value": round(best, 2), "unit": "frames/s", "host_threads": 1,
                    "note": "reference parser on ONE host thread (the streams have one slice per picture and no WPP entry points, so neither "
                            "decoder can parse in parallel) + recording + asynchronous GPU reconstruction + D2H into page-locked picture planes; "
                            "host parsing bounds it (Amdahl). Extra leg, not part of value / e2e"}
    return out


DUMP_SAMPLES = (1 << 18, 1 << 16)  # luma / chroma samples kept per picture: at most 32 x 4 x (2^18 + 2 x 2^16) B = 48 MB


def dump_outputs(eng, step_pics, out_dir):
    """--dump-outputs: what the last timed step of `value` left for its caller in the DPB, i.e. every picture of that step that
    no later picture of the step overwrote, in decode order.  Every plane is sampled at the same seeded positions in each
    picture and written as float32: y.npy (pictures x 2^18), cb.npy and cr.npy (pictures x 2^16), and poc.npy (float64)."""
    last = {p.params.dst_slot: i for i, p in enumerate(step_pics)}
    pics = [step_pics[i] for i in sorted(last.values())]
    rng = np.random.default_rng(0)
    idx, rows = None, [[], [], []]
    for p in pics:
        planes = eng.read_slot(p.params.dst_slot, p.params)
        if idx is None:
            idx = [np.sort(rng.choice(pl.size, min(DUMP_SAMPLES[min(c, 1)], pl.size), replace=False)) for c, pl in enumerate(planes)]
        for c, pl in enumerate(planes):
            rows[c].append(pl.ravel()[idx[c]].astype(np.float32))
    os.makedirs(out_dir, exist_ok=True)
    for c, plane in enumerate(("y", "cb", "cr")):
        np.save(os.path.join(out_dir, plane + ".npy"), np.stack(rows[c]))
    np.save(os.path.join(out_dir, "poc.npy"), np.array([p.params.poc for p in pics], np.float64))


def run_config(name, eng, torch, dist, stream, a, rank, local_rank, world, headline):
    """Runs one bench configuration on this rank's engine: `value` (records resident in HBM, pictures pipelined over the engine's
    streams), the per-stage one-stream pass behind `roofline`, and `e2e` (host records in, pictures out).  Returns the
    config's result dict on rank 0 (None elsewhere)."""
    from libde265_b200 import capi, shard, synth
    cfg = CONFIGS[name]
    width, height, bd = (a.width, a.height, a.bit_depth) if (headline and (a.width, a.height, a.bit_depth) != (W, H, BD)) else (cfg["width"], cfg["height"], cfg["bd"])
    steps = a.steps if headline else max(2, min(a.steps, 4))
    if cfg["kind"] == "ra":
        seq, key_slot, gen_s = build_workload(width, height, bd, seed0=shard.stream_seed(rank) + (0 if headline else 7000))
        ref0 = synth.random_planes(width, height, bd, shard.reference_seed(rank))
        eng.upload_slot(key_slot, seq[0].params, ref0)  # POC 0 reference
    else:
        seq, key_slot, gen_s = build_intra_workload(width, height, bd, seed0=shard.stream_seed(rank) + 3000)
    prepared = [eng.prepare(p) for p in seq]
    h2d_bytes = sum(int(p.pus.nbytes + p.weights.nbytes + p.tus.nbytes + p.coeffs.nbytes + p.slices.nbytes + p.ctbs.nbytes + p.bs_map.nbytes +
                        p.qp_map.nbytes + p.nofilt_map.nbytes) for p in seq) // STEP_VARIANTS
    bps = 2 if bd > 8 else 1
    pic_bytes = width * height * 3 // 2 * bps
    # pinned host output buffers for the e2e leg (a ring of 8: more than the engine keeps pictures in flight)
    dt = torch.uint8 if bps == 1 else torch.int16
    outs = [[torch.empty((height, width), dtype=dt).pin_memory(), torch.empty((height // 2, width // 2), dtype=dt).pin_memory(),
             torch.empty((height // 2, width // 2), dtype=dt).pin_memory()] for _ in range(8)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(n):
            fn()
        eng.join()  # stream 0 waits for the other pipeline streams: e1 marks the completion of every picture
        e1.record(stream)
        e1.synchronize()
        barrier()
        return shard.max_over_ranks(e0.elapsed_time(e1), "cuda")  # the job takes as long as its slowest rank

    counter = {"step": 0}  # shared: the DPB state continues from one step to the next whatever leg runs it

    def step_resident():  # one step; consecutive steps alternate between the workload's variants
        v = counter["step"] % STEP_VARIANTS
        counter["step"] += 1
        for h in prepared[32 * v:32 * (v + 1)]:
            eng.run_prepared(h)

    # e2e goes through the asynchronous submission call (pictures planned by the engine's planner threads, issued in order; the
    # read-back is queued behind its picture); B200_E2E_SYNC=1 measures the one-picture-at-a-time b200_engine_submit_picture instead
    submit = eng.submit if os.environ.get("B200_E2E_SYNC") else eng.submit_async

    def step_e2e():
        v = counter["step"] % STEP_VARIANTS
        counter["step"] += 1
        for i, p in enumerate(seq[32 * v:32 * (v + 1)]):
            submit(p)
            o = outs[i & 7]
            capi.check(eng.lib.b200_engine_read_slot_async(eng.handle, p.params.dst_slot, capi.PlaneArray(*[t.data_ptr() for t in o]),
                                                           capi.StrideArray(*[t.stride(0) * bps for t in o])), "read_slot_async")

    for _ in range(max(3, a.warmup) if headline else 3):
        step_resident()
    eng.sync()
    # ---- value: records resident in HBM, kernels only, pictures pipelined over the engine's streams ----
    clocks = ClockSampler(local_rank)
    clocks.start()
    l0 = eng.launch_count()
    ms_res = timed(step_resident, steps)
    launches = eng.launch_count() - l0
    clk = clocks.stop()
    if headline and a.dump_outputs and rank == 0:
        v = (counter["step"] - 1) % STEP_VARIANTS
        dump_outputs(eng, seq[32 * v:32 * (v + 1)], a.dump_outputs)
    # ---- per-stage kernel times: CUDA events around every stage of every picture on the launching stream.  Stages of
    #      different pictures must not overlap for that, so this pass runs the same steps on ONE stream ----
    eng.enable_timing(True)
    stage_steps = min(steps, 4)
    ms_serial = timed(step_resident, stage_steps)
    stage_ms, n_timed = eng.timing_sum(reset=True)
    eng.enable_timing(False)
    # ---- e2e: host records in, pictures out ----
    # inputs: the record arrays are page-locked and uploaded from where they lie (B200_E2E_PAGEABLE=1: pageable arrays, copied
    # into the engine's pinned staging buffers first)
    pinned = False if os.environ.get("B200_E2E_PAGEABLE") else pin_records(seq, torch)
    for _ in range(4):  # every staging set has reached its final size after the first intra pictures
        step_e2e()
    eng.sync()
    ms_e2e = timed(step_e2e, steps)
    eng.sync()
    if pinned:
        unpin_records(seq, torch)
    for h in prepared:
        eng.free_prepared(h)
    if rank != 0:
        return None

    frames = 32 * steps * world
    fps = frames / (ms_res / 1000.0)
    fps_e2e = frames / (ms_e2e / 1000.0)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    alg = algorithmic_bytes(seq[:32], bd)
    n_inter = sum(1 for p in seq[:32] if len(p.pus))
    per_stage = {}
    for k in ("inter_pred", "recon", "deblock", "sao"):
        ms = stage_ms[k] / max(1, n_timed) * 32  # per step
        gbs = (alg[k] / 1e9) / (ms / 1000.0) if ms > 0 else 0.0
        per_stage[k] = {"ms_per_step": round(ms, 4), "algorithmic_MB_per_step": round(alg[k] / 1e6, 2), "achieved_gbs": round(gbs, 1),
                        "frac": round(gbs / peak, 4)}
    dominant = max(per_stage, key=lambda k: per_stage[k]["ms_per_step"])
    traffic = {}
    try:  # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture
        traffic = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic_per_launch.json")))
    except (OSError, ValueError):
        pass
    mc_kernel = "k_inter_pred_tma" if bd == 8 and not os.environ.get("B200_MC_LEGACY") else ("k_inter_pred8" if bd == 8 else "k_inter_pred<u16>")

    def roof(k):
        launches_per_step = max(1, {"inter_pred": n_inter, "recon": 32, "deblock": 64, "sao": 32}[k])
        return {"kernel": {"inter_pred": mc_kernel, "recon": "k_residual+k_intra", "deblock": "k_deblock<V>+<H>", "sao": "k_sao8" if bd == 8 else "k_sao_prep+k_sao<u16>"}[k],
                "bound": "hbm", "achieved": per_stage[k]["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": per_stage[k]["frac"],
                "traffic": traffic.get(k) if name == "main_ra_4k" else None, "peak_source": peak_src,
                "avg_launch_ms": round(per_stage[k]["ms_per_step"] / launches_per_step, 5),
                "algorithmic_bytes_per_launch": int(alg[k] / launches_per_step),
                "timing": "CUDA events per stage on the launching stream, one-stream pass of %d steps right after the timed region" % stage_steps}

    res = {"value": round(fps, 2), "unit": "frames/s", "steps": steps, "ms_per_step": round(ms_res / steps, 4),
           "dtype": "u8" if bd == 8 else "u16",
           "config": {"workload": cfg["what"] if (width, height, bd) == (cfg["width"], cfg["height"], cfg["bd"]) else
                      f"{width}x{height} {bd}-bit 4:2:0 synthetic command records ({cfg['kind']} structure of {name})",
                      "name": name, "pictures_per_step": 32,
                      "l2_policy": f"per-step working set ({len({p.params.dst_slot for p in seq})} DPB surfaces x {pic_bytes / 1e6:.1f} MB + {STEP_VARIANTS} x 32 record sets) "
                                   "exceeds the 126 MB L2"},
           "e2e": {"value": round(fps_e2e, 2), "unit": "frames/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 32 * pic_bytes,
                   "inputs": "record arrays page-locked (cudaHostRegister), uploaded directly" if pinned else "pageable record arrays through pinned staging",
                   "ms_per_step": round(ms_e2e / steps, 4)},
           "gpu_launches": int(launches), "clocks": clk, "roofline": roof(dominant), "stages": per_stage,
           "one_stream": {"value": round(32 * stage_steps * world / (ms_serial / 1000.0), 2), "unit": "frames/s",
                          "note": "same steps with picture pipelining off (per-stage timing pass)"},
           "workload_gen_s": round(gen_s, 1)}
    if n_inter:
        res["roofline_mc"] = roof("inter_pred")
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="main_ra_4k", choices=sorted(CONFIGS), help="headline workload (default: BASELINE config 3, the one the metric is quoted on)")
    ap.add_argument("--legs", default=None, help="comma-separated extra configs reported under 'legs' (default at 1 GPU: the other two BASELINE configs; 'none' to skip)")
    ap.add_argument("--width", type=int, default=W)
    ap.add_argument("--height", type=int, default=H)
    ap.add_argument("--bit-depth", type=int, default=BD)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of the pictures the last timed step decoded to DIR/*.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg = CONFIGS[a.config]
    custom = (a.width, a.height, a.bit_depth) != (W, H, BD)
    width, height, bd = (a.width, a.height, a.bit_depth) if custom else (cfg["width"], cfg["height"], cfg["bd"])
    legs = [x for x in (a.legs.split(",") if a.legs else ([] if (world > 1 or custom) else [c for c in ("intra1080", "main10_4k", "main_ra_4k") if c != a.config])) if x and x != "none"]

    if a.impl == "reference":
        if rank != 0:
            return 0

        def cpu_arm(w_, h_, bd_, mix):
            reps = 12 if w_ * h_ > 1920 * 1080 else 48
            vals = [cpu_baseline_parallel(w_, h_, bd_, reps, mix=mix) for _ in range(max(1, min(a.steps, 2)))]
            return max(vals, key=lambda v: v["value"])

        best = cpu_arm(width, height, bd, cfg["mix"])
        try:
            real = real_stream_reference()
        except Exception as e:  # informative extra, never fatal
            real = {"error": str(e)[:200]}
        line = {"impl": "reference", "metric": METRIC, "value": best["value"], "unit": "frames/s",
                "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(1000.0 * 32 / best["value"], 3),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8" if bd == 8 else "u16", "data": "synthetic",
                "config": {"workload": cfg["what"], "name": a.config, "pictures_per_step": 32}, "cpu_baseline": best,
                "e2e": {"value": best["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "real_streams": real}
        if legs:
            line["legs"] = {}
            for leg in legs:
                lc = CONFIGS[leg]
                r = cpu_baseline_parallel(lc["width"], lc["height"], lc["bd"], 6 if lc["width"] > 1920 else 24, mix=lc["mix"])
                line["legs"][leg] = {"value": r["value"], "unit": "frames/s", "config": {"workload": lc["what"], "name": leg}, "cpu_baseline": r}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    from libde265_b200.engine import Engine

    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    if world > 1:  # the ranks of one node share its cores: split the host-side threads of the engines between them
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
        cores = effective_cores()[0]
        os.environ.setdefault("B200_ASYNC_THREADS", str(max(2, (cores - 2 * local_world) // local_world)))
        os.environ.setdefault("B200_HOST_THREADS", str(max(2, min(8, cores // local_world))))
    eng = Engine(local_rank)
    stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", local_rank))

    head = run_config(a.config, eng, torch, dist, stream, a, rank, local_rank, world, True)
    leg_res = {}
    for leg in legs:
        try:  # every leg on a fresh engine: surface pool, staging sizes and stream state of one format must not leak into the next
            eng.close()
            eng = Engine(local_rank)
            stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", local_rank))
            leg_res[leg] = run_config(leg, eng, torch, dist, stream, a, rank, local_rank, world, False)
        except Exception as e:  # a leg never takes the headline down
            leg_res[leg] = {"error": str(e)[:300]}
    if rank == 0:
        line = {"metric": METRIC, "value": head["value"], "unit": "frames/s", "n_gpus": world, "steps": a.steps, "warmup": max(3, a.warmup),
                "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": head["dtype"],
                "data": "synthetic", "config": head["config"], "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": head["clocks"],
                "roofline": head["roofline"], "stages": head["stages"], "one_stream": head["one_stream"], "workload_gen_s": head["workload_gen_s"]}
        if "roofline_mc" in head:
            line["roofline_mc"] = head["roofline_mc"]
        if leg_res:
            line["legs"] = leg_res
        try:
            line["real_streams"] = real_stream_b200(eng)
        except Exception as e:  # informative extra, never fatal
            line["real_streams"] = {"error": str(e)[:200]}
        if not a.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_parallel(width, height, bd, 4 if width * height > 1920 * 1080 else 16, mix=cfg["mix"])
        print(json.dumps(line))
    eng.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
