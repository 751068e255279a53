"""Pins every B1-level function of the CPU oracle (oracle/hevc_oracle.c) to the REAL reference function
(oracle/_ref/libref_shim.so -> libde265_ref.so, built from /root/reference by oracle/Makefile), with the
seeds / scenario structure of the reference's own dev-tools tests (SURVEY §4) and the extra cases the
reference leaves unpinned (MC, weighting, DST, IDCT 4/8, transform-skip, 16-bit paths, chroma deblock).
Also checks the reference's SIMD table against its scalar table on the same inputs (what dev-tools/tests do).
Every test also runs without oracle/_ref: the oracle's outputs are then compared with the digests of the reference's outputs
stored in tests/golden/ref_digests.json (oracle_lib.RefDigest)."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib

SHIM = oracle_lib.ref_path("libref_shim.so")

i16p, u8p, u16p, i32p = (C.POINTER(C.c_int16), C.POINTER(C.c_uint8), C.POINTER(C.c_uint16), C.POINTER(C.c_int32))


def P(a, t):
    return a.ctypes.data_as(t)


@pytest.fixture(scope="module")
def ref():
    return C.CDLL(SHIM) if SHIM else None


@pytest.fixture
def digest(request):
    return oracle_lib.ref_digest(request)


@pytest.fixture(scope="module")
def orc():
    lib = oracle_lib.oracle()
    lib.orc_mc_luma.argtypes = [i16p, C.c_int, u16p, C.c_ssize_t] + [C.c_int] * 9
    lib.orc_mc_chroma.argtypes = [i16p, C.c_int, u16p, C.c_ssize_t] + [C.c_int] * 11
    return lib


class XorShift:  # the reference tests' generator (dev-tools/test-transform.cc:44-49)
    def __init__(self, seed):
        self.s = seed & 0xFFFFFFFF

    def next(self):
        s = self.s
        s ^= (s << 13) & 0xFFFFFFFF
        s ^= s >> 17
        s ^= (s << 5) & 0xFFFFFFFF
        self.s = s
        return s


def coeff_scenarios(nT, seed):
    rng = np.random.default_rng(seed)
    x = XorShift(seed)
    sparse = np.zeros(nT * nT, np.int16)
    for _ in range(max(1, nT // 2)):
        sparse[x.next() % (nT * nT // 4 + 1)] = (x.next() % 41) - 20
    dense = rng.integers(-2048, 2049, nT * nT).astype(np.int16)
    full = rng.integers(-32768, 32768, nT * nT).astype(np.int16)
    dc = np.zeros(nT * nT, np.int16)
    dc[0] = 700
    lastrow = np.zeros(nT * nT, np.int16)
    lastrow[-nT:] = rng.integers(-500, 500, nT)
    return [sparse, dense, full, dc, lastrow]


@pytest.mark.parametrize("log2", [2, 3, 4, 5])
@pytest.mark.parametrize("bd", [8, 10, 12])
def test_idct_add(ref, orc, digest, log2, bd):
    nT = 1 << log2
    stride = nT + 17
    rng = np.random.default_rng(0xBEEF1234 + log2 + bd)
    for co in coeff_scenarios(nT, 0xBEEF1234 + log2):
        base = rng.integers(0, 1 << bd, (nT, stride))
        o = base.astype(np.uint16)
        orc.orc_idct_add(P(o, u16p), C.c_ssize_t(stride), nT, P(co, i16p), bd)
        digest.add(o)
        if ref is None:
            continue
        if bd == 8:
            r = base.astype(np.uint8)
            ref.ref_transform_add_8(0, log2, P(r, u8p), P(co, i16p), C.c_ssize_t(stride))
            # the reference's own SIMD-vs-scalar check; the SIMD kernels need 16-byte aligned rows (as in the decoder)
            raw = np.zeros(nT * 64 + 64, np.uint8)
            a0 = (-raw.ctypes.data) % 64
            s = raw[a0:a0 + nT * 64].reshape(nT, 64)
            s[:, :nT] = base[:, :nT]
            ref.ref_transform_add_8(1, log2, P(s, u8p), P(co, i16p), C.c_ssize_t(64))
            assert (s[:, :nT] == r[:, :nT]).all()
        else:
            r = base.astype(np.uint16)
            ref.ref_transform_add_16(0, log2, P(r, u16p), P(co, i16p), C.c_ssize_t(stride), bd)
        assert (o == r).all()  # whole strided buffer, catches out-of-region writes
    digest.check(ref is not None)


@pytest.mark.parametrize("bd", [8, 10])
def test_dst_add(ref, orc, digest, bd):
    stride = 21
    rng = np.random.default_rng(5)
    for co in coeff_scenarios(4, 77):
        base = rng.integers(0, 1 << bd, (4, stride))
        o = base.astype(np.uint16)
        orc.orc_dst4_add(P(o, u16p), C.c_ssize_t(stride), P(co, i16p), bd)
        digest.add(o)
        if ref is None:
            continue
        if bd == 8:
            r = base.astype(np.uint8)
            ref.ref_dst_add_8(0, P(r, u8p), P(co, i16p), C.c_ssize_t(stride))
        else:
            r = base.astype(np.uint16)
            ref.ref_dst_add_16(0, P(r, u16p), P(co, i16p), C.c_ssize_t(stride), bd)
        assert (o == r).all()
    digest.check(ref is not None)


@pytest.mark.parametrize("log2", [2, 3, 4, 5])
def test_dequant(ref, orc, digest, log2):
    # sizes 4..32 x qP 0..51 step 3 x sparsities (dev-tools/test-dequant.cc:51-57), no scaling list
    nT = 1 << log2
    rng = np.random.default_rng(0xD2C0FFEE)
    scale = [40, 45, 51, 57, 64, 72]
    for bd in (8, 10):
        for qp in range(0, 52 + 6 * (bd - 8), 3):
            for nnz in (1, nT, nT * nT // 4, nT * nT):
                pos = rng.choice(nT * nT, nnz, replace=False).astype(np.int16)
                lv = rng.integers(-32768, 32768, nnz).astype(np.int16)
                fact = scale[qp % 6] << (qp // 6)
                bdshift = bd + log2 - 5 - 4
                if fact > 32767:
                    continue  # int64 branch is caller code in the reference (transform.cc:479-487); covered end to end
                o = np.zeros(nT * nT, np.int16)
                r = np.zeros(nT * nT, np.int16)
                orc.orc_dequant(P(o, i16p), P(lv, i16p), P(pos.astype(np.uint16), u16p), nnz, qp, bd, log2, None)
                digest.add(o)
                if ref is not None:
                    ref.ref_dequant(0, P(r, i16p), P(lv, i16p), P(pos, i16p), nnz, fact, 1 << (bdshift - 1), bdshift)
                    assert (o == r).all(), (bd, qp, nnz)
    digest.check(ref is not None)


@pytest.mark.parametrize("log2", [2, 3, 4, 5])
@pytest.mark.parametrize("bd", [8, 10])
def test_transform_skip_and_bypass(ref, orc, digest, log2, bd):
    nT = 1 << log2
    stride = nT + 5
    rng = np.random.default_rng(log2 * 7 + bd)
    co = rng.integers(-3000, 3000, nT * nT).astype(np.int16)
    for rdpcm in (0, 1, 2):
        base = rng.integers(0, 1 << bd, (nT, stride))
        o = base.astype(np.uint16)
        orc.orc_tskip_add(P(o, u16p), C.c_ssize_t(stride), nT, P(co, i16p), bd, rdpcm)
        digest.add(o)
        res = np.zeros(nT * nT, np.int32)
        if ref is not None:
            # reference: residual function + add_residual (transform.cc:566-596)
            if rdpcm == 0:
                ref.ref_tskip_residual(0, P(res, i32p), P(co, i16p), nT, 5 + log2, 20 - bd)
            else:
                ref.ref_rdpcm(0, 1 if rdpcm == 2 else 0, P(res, i32p), P(co, i16p), nT, 5 + log2, 20 - bd)
            r = base.astype(np.uint16)
            ref.ref_add_residual_16(0, P(r, u16p), C.c_ssize_t(stride), P(res, i32p), nT, bd)
            assert (o == r).all(), ("tskip", rdpcm)
        o = base.astype(np.uint16)
        orc.orc_bypass_add(P(o, u16p), C.c_ssize_t(stride), nT, P(co, i16p), bd, rdpcm)
        digest.add(o)
        if ref is not None:
            ref.ref_bypass(0, rdpcm, P(res, i32p), P(co, i16p), nT)
            r = base.astype(np.uint16)
            ref.ref_add_residual_16(0, P(r, u16p), C.c_ssize_t(stride), P(res, i32p), nT, bd)
            assert (o == r).all(), ("bypass", rdpcm)
    digest.check(ref is not None)


def _ref_plane(bd, w, h, seed, extreme):
    rng = np.random.default_rng(seed)
    maxv = (1 << bd) - 1
    if extreme:  # 0/max checkerboards hit the int16 wrap of the V pass (SURVEY App. A.1)
        yy, xx = np.mgrid[0:h, 0:w]
        return (((xx + yy) & 1) * maxv).astype(np.uint16)
    return rng.integers(0, maxv + 1, (h, w)).astype(np.uint16)


@pytest.mark.parametrize("bd", [8, 10])
@pytest.mark.parametrize("extreme", [False, True])
def test_qpel_all_phases(ref, orc, digest, bd, extreme):
    W = H = 96
    plane = _ref_plane(bd, W, H, 0x1234ABCD, extreme)
    p8 = plane.astype(np.uint8)
    for (w, h) in [(4, 8), (8, 4), (8, 8), (12, 16), (16, 16), (24, 32), (32, 8), (64, 64), (48, 64)]:
        for xf in range(4):
            for yf in range(4):
                x0, y0 = 16, 16
                o = np.zeros((h, 64), np.int16)
                orc.orc_mc_luma(P(o, i16p), 64, P(plane, u16p), C.c_ssize_t(W), W, H, x0, y0, xf, yf, w, h, bd)  # mv = frac only
                digest.add(o[:, :w])
                if ref is None:
                    continue
                r = np.zeros((h, 64), np.int16)
                if bd == 8:
                    src = p8[y0:, x0:]
                    ref.ref_put_qpel_8(0, xf, yf, P(r, i16p), C.c_ssize_t(64), C.cast(p8.ctypes.data + y0 * W + x0, u8p), C.c_ssize_t(W), w, h)
                    if w % 8 == 0 or True:
                        s = np.zeros((h, 64), np.int16)
                        ref.ref_put_qpel_8(1, xf, yf, P(s, i16p), C.c_ssize_t(64), C.cast(p8.ctypes.data + y0 * W + x0, u8p), C.c_ssize_t(W), w, h)
                        assert (s[:, :w] == r[:, :w]).all(), ("simd", w, h, xf, yf)
                else:
                    ref.ref_put_qpel_16(0, xf, yf, P(r, i16p), C.c_ssize_t(64), C.cast(plane.ctypes.data + 2 * (y0 * W + x0), u16p), C.c_ssize_t(W), w, h, bd)
                assert (o[:, :w] == r[:, :w]).all(), (w, h, xf, yf)
    digest.check(ref is not None)


@pytest.mark.parametrize("bd", [8, 10])
def test_epel_all_phases(ref, orc, digest, bd):
    W = H = 64  # chroma plane size; luma picture = 128x128
    plane = _ref_plane(bd, W, H, 4321, False)
    p8 = plane.astype(np.uint8)
    for (w, h) in [(2, 4), (4, 2), (4, 4), (6, 8), (8, 8), (16, 4), (32, 32)]:
        for mx in range(8):
            for my in range(8):
                x0, y0 = 8, 8
                o = np.zeros((h, 64), np.int16)
                # luma-unit arguments: xP = 2*x0, mv = eighth-sample fraction only
                orc.orc_mc_chroma(P(o, i16p), 64, P(plane, u16p), C.c_ssize_t(W), 2 * W, 2 * H, 2, 2, 2 * x0, 2 * y0, mx, my, w, h, bd)
                digest.add(o[:, :w])
                if ref is None:
                    continue
                r = np.zeros((h, 64), np.int16)
                if bd == 8:
                    ref.ref_put_epel_8(0, mx, my, P(r, i16p), C.c_ssize_t(64), C.cast(p8.ctypes.data + y0 * W + x0, u8p), C.c_ssize_t(W), w, h)
                else:
                    ref.ref_put_epel_16(0, mx, my, P(r, i16p), C.c_ssize_t(64), C.cast(plane.ctypes.data + 2 * (y0 * W + x0), u16p), C.c_ssize_t(W), w, h, bd)
                assert (o[:, :w] == r[:, :w]).all(), (w, h, mx, my)
    digest.check(ref is not None)


def test_mc_edge_clamping_matches_padded_reference(ref, orc, digest):
    """PUs hanging off all four picture edges: the oracle's coordinate clamping (motion.cc:147-153) must equal the
    reference kernel run on an explicitly edge-replicated copy of the plane."""
    W, H, PAD = 64, 48, 80
    plane = _ref_plane(8, W, H, 99, False)
    padded = np.pad(plane, PAD, mode="edge").astype(np.uint8)
    PW = W + 2 * PAD
    for (x0, y0) in [(-70, -70), (-5, 10), (60, 44), (100, 90), (30, -3), (-8, 47)]:
        for (xf, yf) in [(0, 0), (1, 2), (3, 3), (2, 0), (0, 1)]:
            w, h = 16, 8
            o = np.zeros((h, 64), np.int16)
            orc.orc_mc_luma(P(o, i16p), 64, P(plane, u16p), C.c_ssize_t(W), W, H, 0, 0, 4 * x0 + xf, 4 * y0 + yf, w, h, 8)
            digest.add(o[:, :w])
            if ref is None:
                continue
            r = np.zeros((h, 64), np.int16)
            ref.ref_put_qpel_8(0, xf, yf, P(r, i16p), C.c_ssize_t(64), C.cast(padded.ctypes.data + (y0 + PAD) * PW + x0 + PAD, u8p), C.c_ssize_t(PW), w, h)
            assert (o[:, :w] == r[:, :w]).all(), (x0, y0, xf, yf)
    digest.check(ref is not None)


@pytest.mark.parametrize("bd", [8, 10])
def test_weighted_prediction(ref, orc, digest, bd):
    rng = np.random.default_rng(11)
    w, h, ss = 16, 6, 64
    s1 = rng.integers(-32768, 32768, (h, ss)).astype(np.int16)
    s2 = rng.integers(-32768, 32768, (h, ss)).astype(np.int16)
    s1[0, :4] = [-32768, 32767, 0, 8192]
    ds = 24

    def both(ref_name, ofn, args_o, args_r):
        o = np.zeros((h, ds), np.uint16)
        ofn(P(o, u16p), C.c_ssize_t(ds), *args_o, bd)
        digest.add(o)
        if ref is None:
            return
        if bd == 8:
            r = np.zeros((h, ds), np.uint8)
            getattr(ref, ref_name + "_8")(0, P(r, u8p), C.c_ssize_t(ds), *args_r)
        else:
            r = np.zeros((h, ds), np.uint16)
            getattr(ref, ref_name + "_16")(0, P(r, u16p), C.c_ssize_t(ds), *args_r, bd)
        assert (o == r).all()

    both("ref_put_unweighted", orc.orc_put_unweighted, (P(s1, i16p), ss, w, h), (P(s1, i16p), C.c_ssize_t(ss), w, h))
    both("ref_put_avg", orc.orc_put_avg, (P(s1, i16p), P(s2, i16p), ss, w, h), (P(s1, i16p), P(s2, i16p), C.c_ssize_t(ss), w, h))
    shift1 = max(2, 14 - bd)
    for log2wd in range(shift1, shift1 + 8):
        for (w1, o1, w2, o2) in [(-128, -128, 127, 127), (64, 0, 64, 0), (1, 5, -3, -7), (127, 127, 127, 127), (-128, 0, -128, -128)]:
            o1s, o2s = o1 * (1 << (bd - 8)), o2 * (1 << (bd - 8))
            both("ref_put_weighted", orc.orc_put_weighted, (P(s1, i16p), ss, w, h, w1, o1s, log2wd),
                 (P(s1, i16p), C.c_ssize_t(ss), w, h, w1, o1s, log2wd))
            both("ref_put_bipred", orc.orc_put_weighted_bi, (P(s1, i16p), P(s2, i16p), ss, w, h, w1, o1s, w2, o2s, log2wd),
                 (P(s1, i16p), P(s2, i16p), C.c_ssize_t(ss), w, h, w1, o1s, w2, o2s, log2wd))
    digest.check(ref is not None)


@pytest.mark.parametrize("bd", [8, 10])
def test_intra_all_modes(ref, orc, digest, bd):
    # all 35 modes x nT x cIdx x disableBoundaryFilter (dev-tools/test-intrapred.cc:163-177), + smoothing filter
    x = XorShift(0x1234ABCD)
    for nT in (4, 8, 16, 32):
        for cidx in (0, 1):
            for dis in (0, 1):
                for mode in range(35):
                    for strong_case in (0, 1):
                        raw = np.array([x.next() % (1 << bd) for _ in range(4 * nT + 1)], np.uint16)
                        if strong_case:  # nearly flat border so that strong smoothing triggers for nT=32
                            raw = (np.full(4 * nT + 1, 1 << (bd - 1)) + (np.arange(4 * nT + 1) // 16)).astype(np.uint16)
                        bo = np.zeros(4 * 32 + 8, np.uint16)
                        bo[64 - 2 * nT + 2:64 + 2 * nT + 3] = raw
                        br16 = bo.copy()
                        br8 = bo.astype(np.uint8)
                        co = C.cast(bo.ctypes.data + 2 * 66, u16p)
                        if cidx == 0:
                            orc.orc_intra_filter(co, nT, cidx, mode, 1, bd)
                            digest.add(bo)
                            if ref is None:
                                pass
                            elif bd == 8:
                                ref.ref_intra_filter_8(C.cast(br8.ctypes.data + 66, u8p), nT, cidx, mode, 1)
                                assert (bo == br8).all(), ("filter", nT, mode)
                            else:
                                ref.ref_intra_filter_16(C.cast(br16.ctypes.data + 2 * 66, u16p), nT, cidx, mode, 1, bd)
                                assert (bo == br16).all(), ("filter", nT, mode)
                        stride = nT + 3
                        o = np.zeros((nT, stride), np.uint16)
                        orc.orc_intra_pred(P(o, u16p), C.c_ssize_t(stride), nT, cidx, mode, co, bd, dis)
                        digest.add(o)
                        if ref is None:
                            continue
                        if bd == 8:
                            r = np.zeros((nT, stride), np.uint8)
                            ref.ref_intra_8(0, P(r, u8p), stride, nT, cidx, mode, C.cast(br8.ctypes.data + 66, u8p), dis)
                        else:
                            r = np.zeros((nT, stride), np.uint16)
                            ref.ref_intra_16(0, P(r, u16p), stride, nT, cidx, mode, C.cast(br16.ctypes.data + 2 * 66, u16p), dis, bd)
                        assert (o == r).all(), (nT, cidx, dis, mode)
    digest.check(ref is not None)


@pytest.mark.parametrize("bd", [8, 10])
def test_deblock_segments(ref, orc, digest, bd):
    # all dE/dEp/dEq/filterP/filterQ combos x direction, tc in [1,25] (dev-tools/test-deblk.cc:94-109) + chroma
    x = XorShift(0xDEB10C)
    stride = 16
    for rep in range(30):
        for vertical in (0, 1):
            for dE in (1, 2):
                for dEp in (0, 1):
                    for dEq in (0, 1):
                        for fP in (0, 1):
                            for fQ in (0, 1):
                                tc = (1 + x.next() % 25) * (1 << (bd - 8))
                                base = np.array([(1 << (bd - 1)) + (x.next() % 41) - 20 for _ in range(stride * 12)], np.int32).reshape(12, stride)
                                o = base.astype(np.uint16)
                                off = 4 * stride + 8
                                orc.orc_deblock_luma_seg(C.cast(o.ctypes.data + 2 * off, u16p), C.c_ssize_t(stride), vertical, dE, dEp, dEq, tc, fP, fQ, bd)
                                digest.add(o)
                                if ref is None:
                                    pass
                                elif bd == 8:
                                    r = base.astype(np.uint8)
                                    ref.ref_deblock_luma_8(0, C.cast(r.ctypes.data + off, u8p), C.c_ssize_t(stride), vertical, dE, dEp, dEq, tc, fP, fQ)
                                    s = base.astype(np.uint8)
                                    ref.ref_deblock_luma_8(1, C.cast(s.ctypes.data + off, u8p), C.c_ssize_t(stride), vertical, dE, dEp, dEq, tc, fP, fQ)
                                    assert (s == r).all()
                                else:
                                    r = base.astype(np.uint16)
                                    ref.ref_deblock_luma_16(C.cast(r.ctypes.data + 2 * off, u16p), C.c_ssize_t(stride), vertical, dE, dEp, dEq, tc, fP, fQ, bd)
                                if ref is not None:
                                    assert (o == r).all()
                                o = base.astype(np.uint16)
                                orc.orc_deblock_chroma_seg(C.cast(o.ctypes.data + 2 * off, u16p), C.c_ssize_t(stride), vertical, tc, fP, fQ, bd)
                                digest.add(o)
                                if ref is None:
                                    continue
                                if bd == 8:
                                    r = base.astype(np.uint8)
                                    ref.ref_deblock_chroma_8(0, C.cast(r.ctypes.data + off, u8p), C.c_ssize_t(stride), vertical, tc, fP, fQ)
                                else:
                                    r = base.astype(np.uint16)
                                    ref.ref_deblock_chroma_16(C.cast(r.ctypes.data + 2 * off, u16p), C.c_ssize_t(stride), vertical, tc, fP, fQ, bd)
                                assert (o == r).all()
    digest.check(ref is not None)


# ---- picture-level post-filter drivers (no table entry reaches them) --------------------------------------
POSTFILTER_CASES = [
    # (bit depth, size, log2 CTB, tiles, loop filter across tiles, slices, special_frac (PCM / bypass blocks), picture type)
    (8, (416, 240), 6, (1, 1), True, 1, 0.01, "B"),
    (10, (416, 240), 6, (1, 1), True, 1, 0.01, "B"),
    (8, (320, 200), 5, (1, 1), True, 4, 0.10, "B"),
    (10, (320, 200), 5, (1, 1), True, 4, 0.10, "I"),
    (8, (448, 256), 6, (3, 2), False, 1, 0.05, "B"),
    (10, (448, 256), 6, (2, 3), False, 3, 0.05, "B"),
    (8, (200, 136), 4, (4, 1), True, 2, 0.05, "I"),
    (12, (200, 136), 4, (1, 4), False, 2, 0.05, "B"),
]


@pytest.mark.parametrize("bd,size,log2_ctb,tiles,across,n_slices,special,ptype", POSTFILTER_CASES)
def test_postfilter_drivers_against_reference(ref, digest, bd, size, log2_ctb, tiles, across, n_slices, special, ptype):
    """The oracle's deblocking DRIVER (edge walk, QP averaging, tc / beta from the Q sample's slice, chroma QP mapping,
    pcm / bypass exemptions) and SAO DRIVER (edge + band classes, picture / slice / tile boundary suppression, bypass skip,
    out-of-place input) at 8, 10 and 12 bit against the reference's own edge_filtering_luma / edge_filtering_chroma
    (deblock.cc:412-774, V pass then H pass as deblock.cc:908-946) and apply_sample_adaptive_offset_sequential
    (sao.cc:327-382) run on a synthetic de265_image built from the same records (oracle/ref_shim.cc ref_postfilter)."""
    from libde265_b200 import capi, synth
    W, H = size
    o = oracle_lib.Oracle()
    refs = [synth.random_planes(W, H, bd, s) for s in (7, 8)]
    pic = synth.make_picture(W, H, ptype, seed=900 + bd + n_slices, dst_slot=2, ref_slots=(0, 1) if ptype != "I" else (), bit_depth=bd,
                             log2_ctb=log2_ctb, tiles=tiles, lf_across_tiles=across, n_slices=n_slices, special_frac=special,
                             size_area=(0.1, 0.25, 0.35, 0.3) if log2_ctb == 6 else (0.0, 0.3 if log2_ctb == 5 else 0.0, 0.4, 0.3))
    for s, r in enumerate(refs):
        o.upload_slot(s, pic.params, r)
    stage_out = {}
    for st in (capi.STAGE_RECON, capi.STAGE_DEBLOCK, capi.STAGE_ALL):
        pic.c.params.stop_after_stage = st
        o.reconstruct(pic)
        stage_out[st] = o.read_slot(2, pic.params)
    pic.c.params.stop_after_stage = 0
    o.close()
    dt = np.uint16 if bd > 8 else np.uint8
    # bit 2 = the same drivers dispatching through the reference's SIMD table (what the CPU arm of bench.py times)
    for stages, want in ((1, capi.STAGE_DEBLOCK), (3, capi.STAGE_ALL), (5, capi.STAGE_DEBLOCK), (7, capi.STAGE_ALL)):
        for c in range(3):
            digest.add(stage_out[want][c])
        if ref is None:
            continue
        ref.ref_postfilter.argtypes = [C.POINTER(capi.Picture), capi.PlaneArray, capi.StrideArray, C.c_int, C.c_int, C.c_int]
        planes = [np.ascontiguousarray(p.astype(dt)) for p in stage_out[capi.STAGE_RECON]]
        rc = ref.ref_postfilter(C.byref(pic.c), capi.PlaneArray(*[p.ctypes.data for p in planes]), capi.StrideArray(*[p.strides[0] for p in planes]),
                                stages, tiles[0], tiles[1])
        assert rc == 0
        for c in range(3):
            diff = np.argwhere(planes[c] != stage_out[want][c])
            assert len(diff) == 0, f"stages {stages} plane {c}: {len(diff)} samples differ, first at {diff[0]}"
    digest.check(ref is not None)
    # the filters did something: otherwise the comparison proves nothing
    assert any((a != b).any() for a, b in zip(stage_out[capi.STAGE_RECON], stage_out[capi.STAGE_DEBLOCK]))
    assert any((a != b).any() for a, b in zip(stage_out[capi.STAGE_DEBLOCK], stage_out[capi.STAGE_ALL]))
