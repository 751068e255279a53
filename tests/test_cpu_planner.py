"""Host logic of the engine on CPU (no device needed): b200_plan_picture_host runs the same validation and work-list
building as b200_engine_submit_picture.  Checked here: the MC units tile every PU exactly once, the k_residual classes
partition the non-intra TUs with work, every intra TU is in exactly one task, a task never mixes planes or regions, and —
the property the intra kernel's spin-waits rely on — the task order is TOPOLOGICAL: every neighbour unit a TU may read
(per its availability mask) that an intra TU of this picture produces belongs to the same or an EARLIER task."""
import ctypes as C

import numpy as np
import pytest

from libde265_b200 import capi, synth

AVAIL_CORNER, AVAIL_TOP0 = 16, 17


def plan(lib, pic):
    cp = pic.c
    counts = (C.c_uint32 * 8)()
    n_tu, n_pu = len(pic.tus), len(pic.pus)
    W, H = pic.params.width, pic.params.height
    units = np.zeros(W * H // 32 + 64, np.uint32)
    la, lb, ts = np.zeros(n_tu + 1, np.uint32), np.zeros(n_tu + 1, np.uint32), np.zeros(n_tu + 2, np.uint32)
    p32 = C.POINTER(C.c_uint32)
    rc = lib.b200_plan_picture_host(C.byref(cp), C.byref(counts), units.ctypes.data_as(p32), len(units), la.ctypes.data_as(p32), len(la),
                                    lb.ctypes.data_as(p32), len(lb), ts.ctypes.data_as(p32), len(ts))
    capi.check(rc, "b200_plan_picture_host")
    c = list(counts)
    return dict(units=units[:c[0]], la=la[:c[1]], n_aw=c[2], n_a8=c[3], lb=lb[:c[4]], ts=ts[:c[5] + 1] if c[5] else ts[:0], ref_mask=c[6])


def check_picture(lib, pic):
    r = plan(lib, pic)
    tus, pus = pic.tus, pic.pus
    flags = tus["flags"].astype(int)
    intra = (flags & capi.TU_INTRA) != 0
    work = ((flags & (capi.TU_CBF | capi.TU_PCM)) != 0) & ~intra
    # ---- MC tiles: every predicted PU is cut exactly once into <= 16x16 tiles; the list is sorted into class-pure batches of 8
    #      (class = wide | bi-predicted | tall, kernels_mct.cuh), padded with 0xFFFFFFFF (8-bit pictures; > 8 bit: plain 16x16 tiles) ----
    area = np.zeros(len(pus), np.int64)
    wide_path = pic.params.bit_depth_luma > 8
    real = [int(u) for u in r["units"] if int(u) != 0xFFFFFFFF]
    if not wide_path:
        b = 0
        while b < len(r["units"]):  # batch size by the class of its first tile: 32 tile-list items with the small boxes, else 16
            cls = (int(r["units"][b]) >> 24) & 7
            size = (16 if cls & 5 else 32) >> (1 if cls & 2 else 0)
            batch = [int(u) for u in r["units"][b:b + size]]
            assert len(batch) == size and batch[0] != 0xFFFFFFFF and len({(u >> 24) & 7 for u in batch if u != 0xFFFFFFFF}) == 1
            b += size
    for u in real:
        i, tx, ty = u & 0xFFFFF, (u >> 20) & 3, (u >> 22) & 3
        w, h = int(pus["w"][i]), int(pus["h"][i])
        assert tx * 16 < w and ty * 16 < h
        tw, th = min(16, w - tx * 16), min(16, h - ty * 16)
        area[i] += tw * th
        if not wide_path:
            cls = (u >> 24) & 7
            assert bool(cls & 1) == (tw > 8) and bool(cls & 4) == (th > 8) and bool(cls & 2) == ((int(pus["flags"][i]) & 3) == 3)
    pred = (pus["flags"] & 3) != 0
    assert (area[pred] == pus["w"][pred].astype(np.int64) * pus["h"][pred]).all() and (area[~pred] == 0).all()
    assert len(set(real)) == len(real)
    # ---- k_residual classes ----
    la = r["la"]
    assert sorted(la.tolist()) == np.nonzero(work)[0].tolist()
    l2, pcm = tus["log2_size"][la].astype(int), (flags[la] & capi.TU_PCM) != 0
    assert ((l2[:r["n_aw"]] > 3) | pcm[:r["n_aw"]]).all()
    assert (l2[r["n_aw"]:r["n_aw"] + r["n_a8"]] == 3).all() and (l2[r["n_aw"] + r["n_a8"]:] == 2).all()
    # ---- intra tasks ----
    lb, ts = r["lb"], r["ts"]
    assert sorted(lb.tolist()) == np.nonzero(intra)[0].tolist()
    if not len(lb):
        return 0
    assert ts[0] == 0 and ts[-1] == len(lb) and (np.diff(ts.astype(np.int64)) >= 1).all() and (np.diff(ts.astype(np.int64)) <= 16).all()
    owner = [np.full(((pic.params.height >> (1 if c else 0)) // 4 + 1, (pic.params.width >> (1 if c else 0)) // 4 + 1), -1, np.int64) for c in range(3)]
    task_of = {}
    for t in range(len(ts) - 1):
        members = lb[ts[t]:ts[t + 1]]
        planes = {int(tus["cidx"][i]) for i in members}
        assert len(planes) == 1, f"task {t} mixes planes {sorted(planes)}"
        c0 = planes.pop()
        sh, G = (1 if c0 else 0), 16 >> (1 if c0 else 0)
        rx0, ry0 = (int(tus["x"][members[0]]) << sh) // 16, (int(tus["y"][members[0]]) << sh) // 16
        assert (np.diff(members.astype(np.int64)) > 0).all(), "decode order inside a task"
        for i in members:
            tu = tus[i]
            nT = 1 << int(tu["log2_size"])
            if len(members) > 1:
                assert nT < G and (int(tu["x"]) << sh) // 16 == rx0 and (int(tu["y"]) << sh) // 16 == ry0
            task_of[int(i)] = t
            owner[c0][int(tu["y"]) // 4:(int(tu["y"]) + nT) // 4, int(tu["x"]) // 4:(int(tu["x"]) + nT) // 4] = t
    # ---- topological order ----
    for i, t in task_of.items():
        tu = tus[i]
        c, x4, y4, n4 = int(tu["cidx"]), int(tu["x"]) // 4, int(tu["y"]) // 4, (1 << int(tu["log2_size"])) // 4
        av = int(tu["avail"])
        deps = []
        for k in range(2 * n4):
            if (av >> k) & 1:
                deps.append((y4 + k, x4 - 1))
            if (av >> (AVAIL_TOP0 + k)) & 1:
                deps.append((y4 - 1, x4 + k))
        if (av >> AVAIL_CORNER) & 1:
            deps.append((y4 - 1, x4 - 1))
        for (yy, xx) in deps:
            if 0 <= yy < owner[c].shape[0] and 0 <= xx < owner[c].shape[1] and owner[c][yy, xx] >= 0:
                assert owner[c][yy, xx] <= t, f"TU {i} (task {t}) reads a unit produced by the LATER task {owner[c][yy, xx]}"
    return len(ts) - 1


@pytest.mark.parametrize("kind,size,kw", [("I", (256, 192), {}), ("I", (200, 136), {}), ("B", (320, 192), {}), ("P", (256, 128), dict(special_frac=0.15)),
                                          ("I", (192, 128), dict(log2_ctb=4, size_area=(0.0, 0.0, 0.4, 0.6))), ("I", (192, 128), dict(log2_ctb=5, size_area=(0.0, 0.3, 0.4, 0.3)))])
def test_planner_work_lists(b200lib, kind, size, kw):
    refs = {} if kind == "I" else dict(ref_slots=(0, 1) if kind == "B" else (0,))
    pic = synth.make_picture(size[0], size[1], kind, seed=77, dst_slot=2, **refs, **kw)
    n_tasks = check_picture(b200lib, pic)
    if kind == "I":
        assert n_tasks > 0


def test_planner_rejects_malformed_records(b200lib):
    p = synth.make_picture(64, 64, "P", seed=41, dst_slot=1, ref_slots=(0,))
    p.pus["x"][0] = 62
    with pytest.raises(capi.B200Error):
        plan(b200lib, p)
    q = synth.make_picture(64, 64, "I", seed=42, dst_slot=1)
    q.tus["coeff_off"][-1] = 10 ** 7
    with pytest.raises(capi.B200Error):
        plan(b200lib, q)


def test_planner_on_the_real_1080p_intra_stream(b200lib):
    """The records the reference parser emits for tests/golden/intra1080.h265 (availability masks from the reference's own
    intra_border_computer): ~76k intra TUs in ~23k tasks per picture, task order topological."""
    import os
    import oracle_lib
    from libde265_b200 import de265
    hooked = oracle_lib.ref_path("libde265_hooked.so")
    if hooked is None:
        pytest.skip("oracle/_ref not built")
    dec = de265.Decoder(hooked)
    tasks = []

    class Rec:
        pass

    def sink(pic, planes, strides):
        r = Rec()
        r.c, r.params = pic, pic.params
        r.tus = np.ctypeslib.as_array(C.cast(pic.tus, C.POINTER(C.c_uint8)), shape=(pic.n_tu * 24,)).view(synth.TU_DT).copy()
        r.pus = np.zeros(0, synth.PU_DT)
        tasks.append(check_picture(b200lib, r))
        return 0

    dec.attach(sink)
    n = dec.decode_stream(open(os.path.join(os.path.dirname(__file__), "golden", "intra1080.h265"), "rb").read(), lambda img: None)
    dec.close()
    assert n == 2 and all(t > 20000 for t in tasks)
