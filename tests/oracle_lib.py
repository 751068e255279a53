"""ctypes access to the CPU oracle (oracle/libhevc_oracle.so) and, when present, the real reference
(oracle/_ref/*.so).  TEST INFRASTRUCTURE: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py only."""
import ctypes as C
import hashlib
import json
import os
import subprocess

from libde265_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "libhevc_oracle.so")
REF_DIR = os.path.join(ORACLE_DIR, "_ref")

_orc = None


def build_oracle():
    subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "oracle"])


def oracle():
    global _orc
    if _orc is None:
        if not os.path.exists(ORACLE_SO):
            build_oracle()
        lib = C.CDLL(ORACLE_SO)
        vp = C.c_void_p
        lib.orc_create.restype = vp
        lib.orc_destroy.argtypes = [vp]
        lib.orc_destroy.restype = None
        lib.orc_reconstruct.argtypes = [vp, C.POINTER(capi.Picture)]
        lib.orc_fill_slot.argtypes = [vp, C.c_int, C.POINTER(capi.PicParams), C.c_int, C.c_int]
        lib.orc_upload_slot.argtypes = [vp, C.c_int, C.POINTER(capi.PicParams), capi.PlaneArray, capi.StrideArray]
        lib.orc_read_slot.argtypes = [vp, C.c_int, capi.PlaneArray, capi.StrideArray]
        _orc = lib
    return _orc


def ref_path(name):
    p = os.path.join(REF_DIR, name)
    return p if os.path.exists(p) else None


REF_DIGESTS = os.path.join(ROOT, "tests", "golden", "ref_digests.json")


class RefDigest:
    """SHA-256 over every array one test case compares with the reference, in the order compared.  check() compares it with
    the digest stored under the test's id in tests/golden/ref_digests.json, so the comparison needs no reference build.
    Where oracle/_ref is built the tests also compare each array with the live reference; with REF_DIGESTS_OUT=<json file>
    set, check() then stores the digest (of arrays that all matched the reference) there instead of comparing
    (tests/golden/make_ref_digests.py)."""

    def __init__(self, key):
        self.key, self.h = key, hashlib.sha256()

    def add(self, a):
        import numpy as np
        a = np.ascontiguousarray(a, dtype=np.int32)  # the digest of an 8-bit plane does not depend on its container type
        self.h.update(repr(a.shape).encode())
        self.h.update(a.tobytes())

    def check(self, live):
        got = self.h.hexdigest()
        out = os.environ.get("REF_DIGESTS_OUT")
        if out:
            assert live, "recording a reference digest needs the live reference (oracle/_ref)"
            store = json.load(open(out)) if os.path.exists(out) else {}
            store[self.key] = got
            with open(out, "w") as f:
                json.dump(store, f, indent=0, sort_keys=True)
            return
        want = json.load(open(REF_DIGESTS)).get(self.key)
        assert want is not None, f"no reference digest stored for {self.key}"
        assert got == want, f"{self.key}: the outputs differ from the reference's"


def ref_digest(request):
    """Body of the `digest` fixture of the modules that compare with the reference: one RefDigest per test case."""
    return RefDigest(f"{request.node.module.__name__}::{request.node.name}")


class Oracle:
    """Python wrapper of the CPU restatement's picture replay (orc_*)."""

    def __init__(self):
        self.lib = oracle()
        self.ctx = self.lib.orc_create()

    def close(self):
        if self.ctx:
            self.lib.orc_destroy(self.ctx)
            self.ctx = None

    def reconstruct(self, pic):
        cp = getattr(pic, "c", pic)
        rc = self.lib.orc_reconstruct(self.ctx, C.byref(cp))
        if rc:
            raise RuntimeError(f"orc_reconstruct failed: {rc}")

    def upload_slot(self, slot, params, planes):
        pa = capi.PlaneArray(*[p.ctypes.data for p in planes])
        sa = capi.StrideArray(*[p.strides[0] for p in planes])
        assert self.lib.orc_upload_slot(self.ctx, slot, C.byref(params), pa, sa) == 0

    def fill_slot(self, slot, params, vy, vc):
        assert self.lib.orc_fill_slot(self.ctx, slot, C.byref(params), vy, vc) == 0

    def read_slot(self, slot, params):
        import numpy as np
        dt = np.uint16 if params.bit_depth_luma > 8 else np.uint8
        shapes = [(params.height, params.width)]
        if params.chroma_format_idc:
            shapes += [(params.height // 2, params.width // 2)] * 2
        out = [np.empty(s, dt) for s in shapes]
        ptrs = [o.ctypes.data for o in out] + [None] * (3 - len(out))
        strides = [o.strides[0] for o in out] + [0] * (3 - len(out))
        assert self.lib.orc_read_slot(self.ctx, slot, capi.PlaneArray(*ptrs), capi.StrideArray(*strides)) == 0
        return out


REPLAY_SO = os.path.join(REF_DIR, "libref_replay.so")
_rr = None


def ref_replay_lib():
    """oracle/_ref/libref_replay.so: b200 records replayed through the REFERENCE's own reconstruction functions
    (oracle/ref_replay.cc); None when oracle/_ref was not built / shipped."""
    global _rr
    if _rr is None and os.path.exists(REPLAY_SO):
        lib = C.CDLL(REPLAY_SO)
        vp = C.c_void_p
        lib.rr_create.restype = vp
        lib.rr_create.argtypes = [C.c_int]
        lib.rr_destroy.argtypes = [vp]
        lib.rr_destroy.restype = None
        lib.rr_reconstruct.argtypes = [vp, C.POINTER(capi.Picture)]
        lib.rr_fill_slot.argtypes = [vp, C.c_int, C.POINTER(capi.PicParams), C.c_int, C.c_int]
        lib.rr_upload_slot.argtypes = [vp, C.c_int, C.POINTER(capi.PicParams), capi.PlaneArray, capi.StrideArray]
        lib.rr_read_slot.argtypes = [vp, C.c_int, capi.PlaneArray, capi.StrideArray]
        _rr = lib
    return _rr


class RefReplay(Oracle):
    """Same interface as Oracle, executed by the reference's own code (simd=True: the table de265_acceleration_AUTO selects,
    i.e. SSE4.1 + AVX2 + AVX-512 where the host has them; False: the scalar fallback table)."""

    def __init__(self, simd=True):
        lib = ref_replay_lib()
        if lib is None:
            raise RuntimeError("oracle/_ref/libref_replay.so not built (make -C oracle ref; needs /root/reference)")

        class _Shim:  # present the rr_* entry points under the orc_* names the base class calls
            orc_destroy, orc_reconstruct, orc_upload_slot, orc_fill_slot, orc_read_slot = (lib.rr_destroy, lib.rr_reconstruct, lib.rr_upload_slot,
                                                                                           lib.rr_fill_slot, lib.rr_read_slot)
        self.lib = _Shim
        self.ctx = lib.rr_create(1 if simd else 0)
