"""Boundary B1 (include/b200hevc_dsp.h) on the GPU: every batched DSP-table entry against the REAL reference
function (oracle/_ref/libref_shim.so -> the scalar table of libde265_ref.so), exercised the way the reference's
dev-tools/test-*.cc exercise the SSE table: random blocks, all phases / modes / sizes, 8 and 10 bit.  Bit-exact.  Without
oracle/_ref the GPU's outputs are compared with the digests of the reference's stored in tests/golden/ref_digests.json
(oracle_lib.RefDigest)."""
import ctypes as C

import numpy as np
import pytest

from libde265_b200 import capi
from libde265_b200.dsp import DspTable
import oracle_lib

SHIM = oracle_lib.ref_path("libref_shim.so")
pytestmark = pytest.mark.gpu

i16p, u8p, u16p = C.POINTER(C.c_int16), C.POINTER(C.c_uint8), C.POINTER(C.c_uint16)


def P(a, t, off=0):
    return C.cast(a.ctypes.data + off * a.itemsize, t)


@pytest.fixture(scope="module")
def ref():
    return C.CDLL(SHIM) if SHIM else None


@pytest.fixture
def digest(request):
    return oracle_lib.ref_digest(request)


@pytest.fixture(scope="module")
def dsp():
    d = DspTable(0)
    yield d
    d.close()


def pix(rng, shape, bd, extreme=False):
    hi = (1 << bd) - 1
    a = rng.choice([0, hi], size=shape) if extreme else rng.integers(0, hi + 1, size=shape)
    return a.astype(np.uint8 if bd == 8 else np.uint16)


@pytest.mark.parametrize("bd", [8, 10])
def test_mc_all_phases(ref, dsp, digest, bd):
    rng = np.random.default_rng(1)
    pt = u8p if bd == 8 else u16p
    cases = []
    for luma in (True, False):
        nph = 4 if luma else 8
        for fx in range(nph):
            for fy in range(nph):
                w, h = [(8, 8), (16, 4), (4, 16), (64, 64), (24, 32), (12, 16)][(fx * nph + fy) % 6]
                if not luma:
                    w, h = max(2, w // 2), max(2, h // 2)
                src = pix(rng, (h + 16, w + 16), bd, extreme=(fx + fy) % 5 == 0)
                got = np.zeros((h, w + 3), np.int16)
                exp = np.zeros_like(got)
                st = src.strides[0] // src.itemsize
                dsp.mc(luma, got, src, 8, 8, w, h, fx, fy, bd)
                args = [C.c_int(0), C.c_int(fx), C.c_int(fy), P(exp, i16p), C.c_ssize_t(w + 3), P(src, pt, 8 * st + 8), C.c_ssize_t(st), C.c_int(w), C.c_int(h)]
                if bd > 8:
                    args.append(C.c_int(bd))
                if ref is not None:
                    getattr(ref, f"ref_put_{'qpel' if luma else 'epel'}_{8 if bd == 8 else 16}")(*args)
                cases.append((luma, fx, fy, w, h, got, exp))
    assert dsp.run() == len(cases)
    for luma, fx, fy, w, h, got, exp in cases:
        digest.add(got[:, :w])
        if ref is not None:
            assert (got[:, :w] == exp[:, :w]).all(), f"{'qpel' if luma else 'epel'} phase ({fx},{fy}) {w}x{h}"
    digest.check(ref is not None)


@pytest.mark.parametrize("bd", [8, 10])
def test_weighted_prediction(ref, dsp, digest, bd):
    rng = np.random.default_rng(2)
    pt, suf = (u8p, "8") if bd == 8 else (u16p, "16")
    dt = np.uint8 if bd == 8 else np.uint16
    cases = []
    for k, (w, h) in enumerate([(4, 4), (8, 16), (64, 64), (12, 8), (2, 2), (32, 24)]):
        s1 = rng.integers(-9000, 24000, (h, w + 2)).astype(np.int16)
        s2 = rng.integers(-9000, 24000, (h, w + 2)).astype(np.int16)
        wd = (k % 3) + (14 - bd)  # log2WD = denom + shift1
        w1, o1, w2, o2 = int(rng.integers(-100, 128)), int(rng.integers(-60, 60)), int(rng.integers(-100, 128)), int(rng.integers(-60, 60))
        extra = [C.c_int(bd)] if bd > 8 else []
        for op, name, two, params in ((capi.DSP_PRED_UNI, "ref_put_unweighted_", False, ()), (capi.DSP_PRED_AVG, "ref_put_avg_", True, ()),
                                      (capi.DSP_PRED_WEIGHTED, "ref_put_weighted_", False, (w1, o1, wd)),
                                      (capi.DSP_PRED_WEIGHTED_BI, "ref_put_bipred_", True, (w1, o1, w2, o2, wd))):
            got, exp = np.zeros((h, w + 1), dt), np.zeros((h, w + 1), dt)
            dsp.pred(op, got, s1, s2 if two else None, w, h, bd, params)
            a = [C.c_int(0), P(exp, pt), C.c_ssize_t(w + 1), P(s1, i16p)] + ([P(s2, i16p)] if two else []) + [C.c_ssize_t(w + 2), C.c_int(w), C.c_int(h)]
            if ref is not None:
                getattr(ref, name + suf)(*(a + [C.c_int(v) for v in params] + extra))
            cases.append((name, w, h, got, exp))
    dsp.run()
    for name, w, h, got, exp in cases:
        digest.add(got[:, :w])
        if ref is not None:
            assert (got[:, :w] == exp[:, :w]).all(), f"{name} {w}x{h}"
    digest.check(ref is not None)


@pytest.mark.parametrize("bd", [8, 10])
def test_transform_add(ref, dsp, digest, bd):
    rng = np.random.default_rng(3)
    pt, suf = (u8p, "8") if bd == 8 else (u16p, "16")
    cases = []
    for log2 in (2, 3, 4, 5):
        nT = 1 << log2
        for kind in range(4):
            co = np.zeros(nT * nT, np.int16)
            if kind == 0:
                co[0] = 700
            elif kind == 1:
                co[rng.integers(0, nT * nT, 6)] = rng.integers(-300, 300, 6)
            elif kind == 2:
                co[:] = rng.integers(-2048, 2049, nT * nT)
            else:
                co[:] = rng.integers(-32768, 32768, nT * nT)
            base = np.zeros((nT, 64), np.uint8 if bd == 8 else np.uint16)  # rows 64-element aligned like the reference's planes
            base[:, :nT] = pix(rng, (nT, nT), bd)
            got, exp = base.copy(), base.copy()
            dsp.transform_add(got, co, log2, bd)
            extra = [C.c_int(bd)] if bd > 8 else []
            if ref is not None:
                getattr(ref, "ref_transform_add_" + suf)(C.c_int(0), C.c_int(log2), P(exp, pt), P(co, i16p), C.c_ssize_t(64), *extra)
            cases.append((f"idct{nT} kind {kind}", got, exp))
            if log2 == 2:
                got2, exp2 = base.copy(), base.copy()
                dsp.transform_add(got2, co, 2, bd, dst7=True)
                if ref is not None:
                    getattr(ref, "ref_dst_add_" + suf)(C.c_int(0), P(exp2, pt), P(co, i16p), C.c_ssize_t(64), *extra)
                cases.append((f"dst4 kind {kind}", got2, exp2))
    dsp.run()
    for name, got, exp in cases:
        digest.add(got)
        if ref is not None:
            assert (got == exp).all(), name
    digest.check(ref is not None)


@pytest.mark.parametrize("bd", [8, 10])
def test_intra_prediction(ref, dsp, digest, bd):
    rng = np.random.default_rng(4)
    pt, suf = (u8p, "8") if bd == 8 else (u16p, "16")
    dt = np.uint8 if bd == 8 else np.uint16
    cases = []
    for nT in (4, 8, 16, 32):
        for cidx in (0, 1):
            for mode in range(35):
                border = pix(rng, (4 * nT + 1,), bd)
                got, exp = np.zeros((nT, nT), dt), np.zeros((nT, nT), dt)
                nofilt = int(mode % 7 == 3)
                op = capi.DSP_INTRA_PLANAR if mode == 0 else capi.DSP_INTRA_DC if mode == 1 else capi.DSP_INTRA_ANGULAR
                dsp.intra(op, got, border, nT, cidx, bd, mode, nofilt)
                extra = [C.c_int(bd)] if bd > 8 else []
                if ref is not None:
                    getattr(ref, "ref_intra_" + suf)(C.c_int(0), P(exp, pt), C.c_int(nT), C.c_int(nT), C.c_int(cidx), C.c_int(mode), P(border, pt, 2 * nT), C.c_int(nofilt), *extra)
                cases.append((f"nT {nT} cIdx {cidx} mode {mode}", got, exp))
    dsp.run()
    for name, got, exp in cases:
        digest.add(got)
        if ref is not None:
            assert (got == exp).all(), name
    digest.check(ref is not None)


@pytest.mark.parametrize("bd", [8, 10])
def test_deblock(ref, dsp, digest, bd):
    rng = np.random.default_rng(5)
    pt = u8p if bd == 8 else u16p
    cases = []
    for k in range(200):
        base = (pix(rng, (16, 16), bd) // 8 + (1 << (bd - 1))).astype(np.uint8 if bd == 8 else np.uint16)  # smooth-ish so the filters engage
        got, exp = base.copy(), base.copy()
        vertical, luma = k & 1, (k >> 1) & 1
        tc = int(rng.integers(0, 25)) << (bd - 8)
        fP, fQ = int(rng.integers(0, 2)), int(rng.integers(0, 2))
        if luma:
            params = (int(rng.integers(1, 3)), int(rng.integers(0, 2)), int(rng.integers(0, 2)), tc, fP, fQ)
        else:
            params = (tc, fP, fQ)
        dsp.deblock(bool(luma), got, 8, 8, vertical, bd, params)
        name = f"ref_deblock_{'luma' if luma else 'chroma'}_{8 if bd == 8 else 16}"
        a = ([C.c_int(0)] if bd == 8 else []) + [P(exp, pt, 8 * 16 + 8), C.c_ssize_t(16), C.c_int(vertical)] + [C.c_int(v) for v in params] + ([C.c_int(bd)] if bd > 8 else [])
        if ref is not None:
            getattr(ref, name)(*a)
        cases.append((name, k, got, exp))
    dsp.run()
    for name, k, got, exp in cases:
        digest.add(got)
        if ref is not None:
            assert (got == exp).all(), f"{name} case {k}"
    digest.check(ref is not None)


def test_bad_commands_are_rejected(dsp):
    got = np.zeros((4, 4), np.uint8)
    dsp._add(99, 8, got.ctypes.data, 4)
    with pytest.raises(capi.B200Error):
        dsp.run()
    dsp.transform_add(got, np.zeros(16, np.int16), 7, 8)
    with pytest.raises(capi.B200Error):
        dsp.run()


@pytest.mark.skipif(oracle_lib.ref_path("libde265_b1.so") is None, reason="oracle/_ref/libde265_b1.so not shipped")
def test_reference_decode_loop_on_the_b200_dsp_table_reproduces_golden_md5():
    """The UNMODIFIED reference decoder (its parser, its per-block driver code, its host pictures) with
    init_acceleration_functions_b200 installed (integration/accel_b200.cc): every MC, weighting, inverse transform,
    intra prediction and 8-bit deblocking call of the golden stream runs on the GPU through b200_dsp_run_batch, and the
    output md5 must be the reference's golden md5 (scripts/ci-run.sh:91-92)."""
    import hashlib
    import os
    from libde265_b200 import de265
    from test_cpu_oracle import GOLDEN, GOLDEN_MD5
    dec = de265.Decoder(oracle_lib.ref_path("libde265_b1.so"))
    dec.lib.de265_b200_use_dsp_table.argtypes = [C.c_void_p]
    dec.lib.de265_b200_use_dsp_table.restype = None
    dec.lib.de265_b200_use_dsp_table(dec.ctx)
    md = hashlib.md5()
    n = dec.decode_stream(open(os.path.join(GOLDEN, "girlshy.h265"), "rb").read(), lambda img: [md.update(img.plane_bytes(c)) for c in range(3)])
    dec.close()
    assert n == 75 and md.hexdigest() == GOLDEN_MD5
