"""GPU parity tests (-m gpu): the CUDA engine, called through the C ABI, against the CPU oracle and the
committed golden fixtures.  Bit-exact (integer pixel pipeline): every comparison is array equality."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from libde265_b200 import capi, de265, synth
from libde265_b200.engine import Engine
import oracle_lib
from test_cpu_oracle import GOLDEN, GOLDEN_MD5, load_records

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    e = Engine(0)  # raises (never skips) when the CUDA library or device is missing
    yield e
    e.close()


def md5_planes(planes):
    return hashlib.md5(b"".join(p.tobytes() for p in planes)).hexdigest()


def assert_same(g, o, tag=""):
    for c, (a, b) in enumerate(zip(g, o)):
        if not (a == b).all():
            d = np.argwhere(a != b)
            raise AssertionError(f"{tag} plane {c}: {len(d)} samples differ, first at (x={d[0][1]}, y={d[0][0]}): gpu {a[tuple(d[0])]} != oracle {b[tuple(d[0])]}")


# ---- golden vector: the reference's own known-answer stream ------------------------------------------
def test_girlshy_golden_records_bit_exact(b200lib, eng):
    exp = json.load(open(os.path.join(GOLDEN, "girlshy_expected.json")))
    pics, keep = load_records(b200lib)
    for i, pic in enumerate(pics):
        eng.submit(pic)
        assert md5_planes(eng.read_slot(pic.params.dst_slot, pic.params)) == exp["decode_order_plane_md5"][i], f"picture {i}"


@pytest.mark.skipif(oracle_lib.ref_path("libde265_hooked.so") is None, reason="oracle/_ref not shipped")
def test_girlshy_end_to_end_through_libde265_api(b200lib):
    """de265.h API -> reference parser (B2 hook sites) -> B200 engine -> decoded pictures; md5 of the dec265-style
    output must equal the reference's golden md5 (scripts/ci-run.sh:91-92)."""
    eng = Engine(0)
    dec = de265.Decoder(oracle_lib.ref_path("libde265_hooked.so"))

    def sink(pic, planes, strides):
        eng.submit(pic)
        eng.read_slot_into(pic.params.dst_slot, [planes[0], planes[1], planes[2]], [strides[0], strides[1], strides[2]])
        return 0

    dec.attach(sink)
    md = hashlib.md5()
    n = dec.decode_stream(open(os.path.join(GOLDEN, "girlshy.h265"), "rb").read(), lambda img: [md.update(img.plane_bytes(c)) for c in range(3)])
    dec.close()
    assert n == 75 and md.hexdigest() == GOLDEN_MD5
    assert eng.launch_count() > 75 * 4
    eng.close()


@pytest.mark.parametrize("name", ["intra1080", "intra4k"])
@pytest.mark.skipif(oracle_lib.ref_path("libde265_hooked.so") is None, reason="oracle/_ref not shipped")
def test_real_intra_stream_end_to_end(b200lib, name):
    """BASELINE config 2's size (1080p intra) and the 4K size on REAL bitstreams (made with the reference's own encoder,
    tests/golden/make_intra_streams.py): reference parser -> records -> B200 engine; md5 of the output must equal the
    unmodified reference decoder's."""
    exp = json.load(open(os.path.join(GOLDEN, name + "_expected.json")))
    eng = Engine(0)
    dec = de265.Decoder(oracle_lib.ref_path("libde265_hooked.so"))

    def sink(pic, planes, strides):
        eng.submit(pic)
        eng.read_slot_into(pic.params.dst_slot, [planes[0], planes[1], planes[2]], [strides[0], strides[1], strides[2]])
        return 0

    dec.attach(sink)
    md = hashlib.md5()
    n = dec.decode_stream(open(os.path.join(GOLDEN, name + ".h265"), "rb").read(), lambda img: [md.update(img.plane_bytes(c)) for c in range(3)])
    dec.close()
    eng.close()
    assert n == exp["pictures"] and md.hexdigest() == exp["md5_of_all_planes_in_output_order"]


@pytest.mark.parametrize("lag,queued", [(0, False), (1, False), (1, True)])
@pytest.mark.skipif(oracle_lib.ref_path("libde265_hooked.so") is None, reason="oracle/_ref not shipped")
def test_girlshy_through_the_acceleration_code(b200lib, monkeypatch, lag, queued):
    """The drop-in switch itself: de265_set_parameter_int(ctx, DE265_DECODER_PARAM_ACCELERATION_CODE, de265_acceleration_B200)
    on a libde265 built with the binding of INTEGRATION.md — no sink, no Python in the data path: the decoder owns a B200 engine,
    submits every picture asynchronously at picture end and awaits the read-back when the picture is handed out.  Golden md5 of
    scripts/ci-run.sh:91-92, with the dec265 loop (lag 0) and with pictures fetched one de265_decode call late (lag 1); `queued`:
    the backend queues the pictures (b200_engine_submit_picture_async, ring of recorders, tickets) instead of planning them in the hook."""
    if queued:
        monkeypatch.setenv("B200_HOOK_ASYNC", "1")
    dec = de265.Decoder(oracle_lib.ref_path("libde265_hooked.so"))
    dec.select_b200()
    md = hashlib.md5()
    n = dec.decode_stream(open(os.path.join(GOLDEN, "girlshy.h265"), "rb").read(), lambda img: [md.update(img.plane_bytes(c)) for c in range(3)], lag=lag)
    dec.close()
    assert n == 75 and md.hexdigest() == GOLDEN_MD5


@pytest.mark.skipif(oracle_lib.ref_path("libde265_hooked.so") is None or oracle_lib.ref_path("libde265_ref.so") is None, reason="oracle/_ref not shipped")
def test_concatenated_intra_streams_through_the_acceleration_code(b200lib):
    """The real 1080p intra stream three times back to back (every copy starts with its own parameter sets and an IDR picture)
    through the asynchronous built-in backend, pictures fetched one call late so that parsing overlaps the GPU: the same
    pictures as the unmodified reference decoder produces from the same bytes."""
    data = open(os.path.join(GOLDEN, "intra1080.h265"), "rb").read() * 3
    want, got = [], []
    ref = de265.Decoder(oracle_lib.ref_path("libde265_ref.so"))
    ref.decode_stream(data, lambda img: want.append(hashlib.md5(b"".join(img.plane_bytes(c) for c in range(3))).hexdigest()))
    ref.close()
    dec = de265.Decoder(oracle_lib.ref_path("libde265_hooked.so"))
    dec.select_b200()
    dec.decode_stream(data, lambda img: got.append(hashlib.md5(b"".join(img.plane_bytes(c) for c in range(3))).hexdigest()), lag=1)
    dec.close()
    assert len(want) == 6 and got == want


# ---- synthetic pictures vs the oracle -----------------------------------------------------------------
def run_sequence(eng, orc, W, H, bd, log2_ctb=6, stages=False, **kw):
    ref = synth.random_planes(W, H, bd, 99)
    pics = [synth.make_picture(W, H, "I", seed=11, dst_slot=0, bit_depth=bd, log2_ctb=log2_ctb, **kw)]
    eng.upload_slot(5, pics[0].params, ref)
    orc.upload_slot(5, pics[0].params, ref)
    pics.append(synth.make_picture(W, H, "P", seed=12, dst_slot=1, ref_slots=(0, 5), bit_depth=bd, log2_ctb=log2_ctb, **kw))
    pics.append(synth.make_picture(W, H, "B", seed=13, dst_slot=2, ref_slots=(0, 1, 5), bit_depth=bd, log2_ctb=log2_ctb, **kw))
    pics.append(synth.make_picture(W, H, "B", seed=14, dst_slot=3, ref_slots=(0, 1, 2), weighted=True, bit_depth=bd, log2_ctb=log2_ctb, **kw))
    for i, p in enumerate(pics):
        for st in ((capi.STAGE_INTER_PRED, capi.STAGE_RECON, capi.STAGE_DEBLOCK, capi.STAGE_ALL) if stages else (capi.STAGE_ALL,)):
            p.c.params.stop_after_stage = st
            eng.submit(p)
            orc.reconstruct(p)
            assert_same(eng.read_slot(p.params.dst_slot, p.params), orc.read_slot(p.params.dst_slot, p.params), f"pic {i} stage {st}")
        p.c.params.stop_after_stage = 0


@pytest.mark.parametrize("bd", [8, 10])
def test_synthetic_sequence_every_stage(eng, oracle_mod, bd):
    orc = oracle_mod.Oracle()
    run_sequence(eng, orc, 416, 240, bd, stages=True)
    orc.close()


@pytest.mark.parametrize("size", [(8, 8), (16, 8), (72, 40), (64, 64), (200, 136), (1288, 8)])
def test_ragged_and_tiny_pictures(eng, oracle_mod, size):
    """Pictures that are not a multiple of the CTB size, down to a single minimum CB."""
    orc = oracle_mod.Oracle()
    run_sequence(eng, orc, size[0], size[1], 8)
    orc.close()


@pytest.mark.parametrize("log2_ctb", [4, 5])
def test_small_ctb_sizes(eng, oracle_mod, log2_ctb):
    orc = oracle_mod.Oracle()
    run_sequence(eng, orc, 208, 120, 8, log2_ctb=log2_ctb, size_area=(0.0, 0.3 if log2_ctb == 5 else 0.0, 0.4, 0.3))
    orc.close()


def test_multi_slice_scaling_list_no_filters(eng, oracle_mod):
    orc = oracle_mod.Oracle()
    run_sequence(eng, orc, 320, 192, 8, n_slices=4, scaling_list=True)
    run_sequence(eng, orc, 320, 192, 10, deblock=False, sao=False)
    run_sequence(eng, orc, 320, 192, 8, special_frac=0.15, cbf_prob=0.9)  # many PCM / bypass / transform-skip blocks
    orc.close()


def test_1080p_intra_and_4k_b_frame(eng, oracle_mod):
    """BASELINE configs 2 and 3 at full size against the oracle (one picture each; the oracle needs a few seconds)."""
    orc = oracle_mod.Oracle()
    p = synth.make_picture(1920, 1080, "I", seed=21, dst_slot=0)
    eng.submit(p)
    orc.reconstruct(p)
    assert_same(eng.read_slot(0, p.params), orc.read_slot(0, p.params), "1080p intra")
    W, H = 3840, 2160
    refs = [synth.random_planes(W, H, 8, s) for s in (1, 2)]
    b = synth.make_picture(W, H, "B", seed=22, dst_slot=2, ref_slots=(0, 1))
    for s, r in enumerate(refs):
        eng.upload_slot(s, b.params, r)
        orc.upload_slot(s, b.params, r)
    eng.submit(b)
    orc.reconstruct(b)
    assert_same(eng.read_slot(2, b.params), orc.read_slot(2, b.params), "4K B")
    orc.close()


def test_4k_main10_against_oracle_and_prepared_path(eng, oracle_mod):
    """BASELINE config 4 at full size (3840x2160, 10 bit): one B picture (explicit weights on, both lists, far MVs) and one I
    picture against the oracle, sample by sample; then the size-independent properties on top: replaying the same records is
    idempotent and the prepared (HBM-resident) path equals the submit path."""
    W, H = 3840, 2160
    orc = oracle_mod.Oracle()
    refs = [synth.random_planes(W, H, 10, s) for s in (3, 4)]
    b = synth.make_picture(W, H, "B", seed=23, dst_slot=2, ref_slots=(0, 1), bit_depth=10, weighted=True)
    for s, r in enumerate(refs):
        eng.upload_slot(s, b.params, r)
        orc.upload_slot(s, b.params, r)
    eng.submit(b)
    orc.reconstruct(b)
    got = eng.read_slot(2, b.params)
    assert_same(got, orc.read_slot(2, b.params), "4K Main10 B")
    first = md5_planes(got)
    eng.submit(b)
    assert md5_planes(eng.read_slot(2, b.params)) == first
    h = eng.prepare(b)
    eng.fill_slot(2, b.params, 0, 0)
    eng.run_prepared(h)
    assert md5_planes(eng.read_slot(2, b.params)) == first
    eng.free_prepared(h)
    i = synth.make_picture(W, H, "I", seed=24, dst_slot=3, bit_depth=10)
    eng.submit(i)
    orc.reconstruct(i)
    assert_same(eng.read_slot(3, i.params), orc.read_slot(3, i.params), "4K Main10 I")
    orc.close()


@pytest.mark.parametrize("bd", [8, 10])
def test_rdpcm_rotation_and_large_transform_skip(eng, oracle_mod, bd):
    """RExt residual variants the hooks can record (transform.cc:402-448, 548-596): horizontal / vertical RDPCM on
    transform-skip and bypass TUs of every size, coefficient rotation on 4x4 TUs of intra CUs, transform skip up to 32x32;
    stage by stage against the oracle (whose RDPCM / rotation / skip functions are pinned to the reference's table entries
    in test_oracle_vs_ref.py)."""
    orc = oracle_mod.Oracle()
    run_sequence(eng, orc, 320, 192, bd, stages=True, special_frac=0.2, cbf_prob=0.9, rdpcm_frac=0.5, rotate_frac=0.5, tskip_max_log2=5)
    orc.close()


@pytest.mark.parametrize("bd,tiles,across,n_slices", [(8, (3, 2), False, 1), (8, (2, 3), True, 3), (10, (4, 1), False, 2), (8, (1, 4), False, 4)])
def test_tiles(eng, oracle_mod, bd, tiles, across, n_slices):
    """Multi-tile pictures: CTBs recorded in tile-scan order, intra availability cut at tile borders (intrapred.h:488-503),
    no deblocking edge and no SAO neighbour across a tile border when loop_filter_across_tiles is off (deblock.cc:196-203,
    sao.cc:157-163); with several slices on top.  Stage by stage against the oracle."""
    orc = oracle_mod.Oracle()
    run_sequence(eng, orc, 448, 256, bd, stages=True, tiles=tiles, lf_across_tiles=across, n_slices=n_slices)
    run_sequence(eng, orc, 200, 136, bd, log2_ctb=4, tiles=tiles, lf_across_tiles=across, n_slices=n_slices, size_area=(0.0, 0.0, 0.5, 0.5))
    orc.close()


def test_pipelined_streams_match_serial_and_oracle(oracle_mod):
    """Picture pipelining over several CUDA streams (per-slot event ordering) must not change a single sample: a
    hierarchical-B sequence with a small slot ring (every hazard kind: RAW on references, WAR/WAW on reused slots),
    submitted back to back without host syncs, on 1 and on 4 streams, against the oracle."""
    W, H = 256, 128
    order = [("I", 0, ()), ("P", 8, (0,)), ("B", 4, (0, 8)), ("B", 2, (0, 4)), ("B", 1, (0, 2)), ("B", 3, (2, 4)), ("B", 6, (4, 8)),
             ("B", 5, (4, 6)), ("B", 7, (6, 8)), ("P", 16, (8,)), ("B", 12, (8, 16)), ("B", 10, (8, 12)), ("B", 9, (8, 10)),
             ("B", 11, (10, 12)), ("B", 14, (12, 16)), ("B", 13, (12, 14)), ("B", 15, (14, 16)), ("I", 24, ())]
    ring = 10  # slots poc % 10: 16 overwrites 6, 12 overwrites 2, ...
    pics = [synth.make_picture(W, H, t, seed=500 + poc, dst_slot=poc % ring, ref_slots=tuple(r % ring for r in refs)) for t, poc, refs in order]
    orc = oracle_mod.Oracle()
    expect = []
    for p in pics:
        orc.reconstruct(p)
        expect.append(md5_planes(orc.read_slot(p.params.dst_slot, p.params)))
    orc.close()
    for n, submit_async in ((1, False), (4, False), (8, True)):  # the asynchronous call: planner threads + in-order sequencer, reads queued
        e = Engine(0)
        e.set_streams(n)
        bufs = [[np.empty((H, W), np.uint8), np.empty((H // 2, W // 2), np.uint8), np.empty((H // 2, W // 2), np.uint8)] for _ in pics]
        for rep in range(3):  # repeated: later rounds overwrite slots that earlier pictures still read
            for p, b in zip(pics, bufs):
                (e.submit_async if submit_async else e.submit)(p)
                capi.check(e.lib.b200_engine_read_slot_async(e.handle, p.params.dst_slot, capi.PlaneArray(*[x.ctypes.data for x in b]),
                                                             capi.StrideArray(*[x.strides[0] for x in b])), "read_slot_async")
            e.sync()
            got = [md5_planes(b) for b in bufs]
            assert got == expect, f"{n} stream(s), round {rep}: pictures {[i for i, (g, x) in enumerate(zip(got, expect)) if g != x]} differ"
        e.close()


def test_missing_reference_and_fill_slot(eng, oracle_mod):
    orc = oracle_mod.Oracle()
    W, H = 128, 64
    p = synth.make_picture(W, H, "B", seed=31, dst_slot=3, ref_slots=(7, 9))  # slot 9 never written -> mid-grey prediction
    eng2 = Engine(0)
    eng2.fill_slot(7, p.params, 77, 200)
    orc.fill_slot(7, p.params, 77, 200)
    eng2.submit(p)
    orc.reconstruct(p)
    assert_same(eng2.read_slot(3, p.params), orc.read_slot(3, p.params), "missing ref")
    eng2.close()
    orc.close()


def test_malformed_records_are_rejected(eng):
    p = synth.make_picture(64, 64, "P", seed=41, dst_slot=1, ref_slots=(0,))
    p.pus["x"][0] = 62  # not on the 4-sample grid / outside
    with pytest.raises(capi.B200Error):
        eng.submit(p)
    q = synth.make_picture(64, 64, "I", seed=42, dst_slot=1)
    q.tus["coeff_off"][-1] = 10 ** 7
    with pytest.raises(capi.B200Error):
        eng.submit(q)
    r = synth.make_picture(64, 64, "I", seed=43, dst_slot=1)
    r.c.params.chroma_format_idc = 3
    with pytest.raises(capi.B200Error):
        eng.submit(r)
    # the asynchronous call reports a queued picture's error at the next flush; the pictures around it are not affected
    ok = synth.make_picture(64, 64, "I", seed=44, dst_slot=2)
    eng.submit_async(ok)
    eng.submit_async(q)
    eng.submit_async(ok)
    with pytest.raises(capi.B200Error):
        eng.flush()
    eng.flush()  # the error was consumed
    eng.sync()


def test_unsatisfiable_intra_dependencies_are_reported_not_hung(monkeypatch):
    """Availability bits that lie outside the picture are rejected on the host; bits that name a unit reconstructed LATER (here two
    16x16+ TUs that wait for each other) cannot be seen on the host cheaply: k_intra's dependency wait is bounded, the picture is
    flagged and the next synchronisation point returns B200_ERR_INVALID instead of hanging the stream."""
    p = synth.make_picture(128, 128, "I", seed=40, dst_slot=1)
    t = p.tus
    pair = None
    for i in range(len(t)):
        a = t[i]
        nT = 1 << int(a["log2_size"])
        if a["cidx"] != 0 or nT < 16 or a["x"] % (2 * nT) != nT or a["y"] % (2 * nT) != 0 or a["y"] + 2 * nT > 128:
            continue
        for j in range(i + 1, len(t)):
            b = t[j]
            if b["cidx"] == 0 and b["log2_size"] == a["log2_size"] and b["x"] == a["x"] - nT and b["y"] == a["y"] + nT:
                pair = (i, j, nT)
                break
        if pair:
            break
    assert pair, "no top-right / bottom-left TU pair in the synthetic picture"
    i, j, nT = pair
    q = nT // 4
    below_left = sum(1 << k for k in range(q, 2 * q))
    keep = int(t["avail"][i])
    t["avail"][0] |= 1  # TU 0 sits at x = 0: a left neighbour is outside the picture
    e0 = Engine(0)
    with pytest.raises(capi.B200Error):
        e0.submit(p)
    t["avail"][0] &= ~np.uint64(1)
    e0.close()
    t["avail"][i] = keep | below_left                                  # A waits for B, which comes later ...
    t["avail"][j] = int(t["avail"][j]) | (below_left << 17)            # ... and B (legitimately) waits for A, its top-right neighbour
    monkeypatch.setenv("B200_INTRA_SPIN_LIMIT_MS", "50")
    e = Engine(0)
    e.submit(p)
    with pytest.raises(capi.B200Error, match="dependency wait"):
        e.sync()
    t["avail"][i] = keep
    e.submit(p)  # the engine keeps working
    e.sync()
    e.close()


def test_records_uploaded_straight_from_pinned_arrays(eng, oracle_mod):
    """B200_PIC_RECORDS_PINNED: the engine uploads the raw record arrays from the caller's page-locked memory (no staging copy);
    same pictures as through the staging path, synchronous and asynchronous submission."""
    lib = eng.lib
    W, H = 320, 192
    base = [synth.make_picture(W, H, "I", seed=71, dst_slot=0), synth.make_picture(W, H, "P", seed=72, dst_slot=1, ref_slots=(0,)),
            synth.make_picture(W, H, "B", seed=73, dst_slot=2, ref_slots=(0, 1), weighted=True)]
    orc = oracle_mod.Oracle()
    expect = []
    for p in base:
        orc.reconstruct(p)
        expect.append(orc.read_slot(p.params.dst_slot, p.params))
    orc.close()
    blocks = []

    def pinned_copy(a):
        if a is None or not len(a):
            return a
        ptr = lib.b200_host_alloc(a.nbytes)
        assert ptr
        blocks.append(ptr)
        out = np.frombuffer((C.c_uint8 * a.nbytes).from_address(ptr), dtype=a.dtype, count=len(a))
        out[:] = a
        return out

    pics = []
    for p in base:
        q = synth.SynthPicture(p.params, *[pinned_copy(getattr(p, n)) for n in ("pus", "weights", "tus", "coeffs", "slices", "ctbs", "bs_map", "qp_map", "nofilt_map")])
        q.c.params.flags |= capi.PIC_RECORDS_PINNED
        pics.append(q)
    for use_async in (False, True):
        e = Engine(0)
        for q in pics:
            (e.submit_async if use_async else e.submit)(q)
        e.sync()
        for q, x in zip(pics, expect):
            assert_same(e.read_slot(q.params.dst_slot, q.params), x, f"pinned records, async={use_async}")
        e.close()
    for ptr in blocks:
        lib.b200_host_free(ptr)


def test_empty_picture(eng, oracle_mod):
    """No PUs and no TUs: every stage must cope with empty work lists (samples no record covers keep the slot's
    content; with SAO on they would come from the scratch surface, which only a malformed stream can expose)."""
    orc = oracle_mod.Oracle()
    p = synth.make_picture(64, 64, "I", seed=44, dst_slot=1, sao=False)
    e = synth.SynthPicture(p.params, p.pus[:0], p.weights, p.tus[:0], p.coeffs[:0], p.slices, p.ctbs, p.bs_map, p.qp_map, p.nofilt_map)
    eng.fill_slot(1, p.params, 50, 60)
    orc.fill_slot(1, p.params, 50, 60)
    eng.submit(e)
    orc.reconstruct(e)
    assert_same(eng.read_slot(1, p.params), orc.read_slot(1, p.params), "empty")
    orc.close()
