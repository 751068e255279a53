"""The record-replay executor over the REFERENCE's own reconstruction functions (oracle/ref_replay.cc ->
oracle/_ref/libref_replay.so: generate_inter_prediction_samples, decode_intra_prediction, scale_coefficients,
edge_filtering_luma/chroma, apply_sample_adaptive_offset_sequential on the reference's scalar and SIMD tables) against the
CPU oracle, picture by picture and stage by stage.  This pins the oracle's PICTURE-LEVEL driver (PU loop with edge clamping
and all weighting modes, intra availability from slices / tiles / z-scan, TU loop, both post filters) to the reference at
8 and 10 bit — not only its per-block functions — and validates the CPU arm bench.py times.  Without oracle/_ref the oracle's
pictures are compared with the digests of the reference's stored in tests/golden/ref_digests.json (oracle_lib.RefDigest)."""
import hashlib
import json
import os

import numpy as np
import pytest

import oracle_lib
from libde265_b200 import capi, synth
from test_cpu_oracle import GOLDEN, load_records

LIVE = oracle_lib.ref_replay_lib() is not None


@pytest.fixture
def digest(request):
    return oracle_lib.ref_digest(request)


def same(a, b, tag):
    for c, (x, y) in enumerate(zip(a, b)):
        d = np.argwhere(x != y)
        assert len(d) == 0, f"{tag} plane {c}: {len(d)} samples differ, first at (x={d[0][1]}, y={d[0][0]}): reference {x[tuple(d[0])]} != oracle {y[tuple(d[0])]}"


def run_sequence(digest, W, H, bd, simd, log2_ctb=6, stages=True, **kw):
    orc, ref = oracle_lib.Oracle(), oracle_lib.RefReplay(simd=simd) if LIVE else None
    planes = synth.random_planes(W, H, bd, 99)
    pics = [synth.make_picture(W, H, "I", seed=11, dst_slot=0, bit_depth=bd, log2_ctb=log2_ctb, **kw)]
    for e in [orc] + ([ref] if LIVE else []):
        e.upload_slot(5, pics[0].params, planes)
    pics.append(synth.make_picture(W, H, "P", seed=12, dst_slot=1, ref_slots=(0, 5), bit_depth=bd, log2_ctb=log2_ctb, **kw))
    pics.append(synth.make_picture(W, H, "B", seed=13, dst_slot=2, ref_slots=(0, 1, 5), bit_depth=bd, log2_ctb=log2_ctb, **kw))
    pics.append(synth.make_picture(W, H, "B", seed=14, dst_slot=3, ref_slots=(0, 1, 2), weighted=True, bit_depth=bd, log2_ctb=log2_ctb, **kw))
    for i, p in enumerate(pics):
        for st in ((capi.STAGE_INTER_PRED, capi.STAGE_RECON, capi.STAGE_DEBLOCK, capi.STAGE_ALL) if stages else (capi.STAGE_ALL,)):
            p.c.params.stop_after_stage = st
            orc.reconstruct(p)
            got = orc.read_slot(p.params.dst_slot, p.params)
            for c in got:
                digest.add(c)
            if LIVE:
                ref.reconstruct(p)
                same(ref.read_slot(p.params.dst_slot, p.params), got, f"pic {i} stage {st}")
        p.c.params.stop_after_stage = 0
    orc.close()
    if LIVE:
        ref.close()


@pytest.mark.parametrize("simd", [False, True])
@pytest.mark.parametrize("bd", [8, 10])
def test_replay_matches_oracle_every_stage(digest, bd, simd):
    run_sequence(digest, 416, 240, bd, simd)
    digest.check(LIVE)


@pytest.mark.parametrize("simd", [False, True])
def test_replay_ragged_sizes_and_small_ctbs(digest, simd):
    for size in ((8, 8), (72, 40), (200, 136), (1288, 8)):
        run_sequence(digest, size[0], size[1], 8, simd, stages=False)
    run_sequence(digest, 208, 120, 8, simd, log2_ctb=4, stages=False, size_area=(0.0, 0.0, 0.5, 0.5))
    run_sequence(digest, 208, 120, 10, simd, log2_ctb=5, stages=False, size_area=(0.0, 0.3, 0.4, 0.3))
    digest.check(LIVE)


@pytest.mark.parametrize("simd", [False, True])
def test_replay_slices_scaling_lists_special_blocks_tiles(digest, simd):
    run_sequence(digest, 320, 192, 8, simd, n_slices=4, scaling_list=True)
    run_sequence(digest, 320, 192, 10, simd, deblock=False, sao=False, stages=False)
    run_sequence(digest, 320, 192, 8, simd, special_frac=0.15, cbf_prob=0.9)
    run_sequence(digest, 320, 192, 10, simd, special_frac=0.2, cbf_prob=0.9, rdpcm_frac=0.5, rotate_frac=0.5, tskip_max_log2=5)
    run_sequence(digest, 448, 256, 8, simd, tiles=(3, 2), lf_across_tiles=False)
    run_sequence(digest, 448, 256, 10, simd, tiles=(2, 3), lf_across_tiles=True, n_slices=3)
    digest.check(LIVE)


def test_replay_missing_reference_and_fill(digest):
    orc = oracle_lib.Oracle()
    p = synth.make_picture(128, 64, "B", seed=31, dst_slot=3, ref_slots=(7, 9))  # slot 9 never written -> mid-grey prediction
    orc.fill_slot(7, p.params, 77, 200)
    orc.reconstruct(p)
    got = orc.read_slot(3, p.params)
    for c in got:
        digest.add(c)
    orc.close()
    if LIVE:
        ref = oracle_lib.RefReplay(simd=True)
        ref.fill_slot(7, p.params, 77, 200)
        ref.reconstruct(p)
        same(ref.read_slot(3, p.params), got, "missing reference")
        ref.close()
    digest.check(LIVE)


@pytest.mark.parametrize("simd", [False, True])
@pytest.mark.skipif(not LIVE, reason="oracle/_ref/libref_replay.so not built (needs the reference sources)")
def test_replay_reproduces_the_golden_stream(b200lib, simd):
    """Records of the reference's own known-answer stream (recorded by the hooked reference parser): the replay through the
    reference's functions must land on the per-picture md5s of the unmodified reference decoder."""
    exp = json.load(open(os.path.join(GOLDEN, "girlshy_expected.json")))
    pics, keep = load_records(b200lib)
    ref = oracle_lib.RefReplay(simd=simd)
    for i, pic in enumerate(pics):
        ref.reconstruct(pic)
        got = hashlib.md5(b"".join(p.tobytes() for p in ref.read_slot(pic.params.dst_slot, pic.params))).hexdigest()
        assert got == exp["decode_order_plane_md5"][i], f"picture {i}"
    ref.close()
