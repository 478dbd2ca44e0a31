"""ctypes wrapper over tests/emul/libemul_s*.so — TEST INFRASTRUCTURE.

The emulator runs the PRODUCT's host driver and __host__ __device__ DP core on the CPU with the
CUDA kernel's tile/lane/round structure emulated sequentially; the CPU-only tests fuzz it against
the oracle.  It exports the product's C ABI under the emul_ prefix."""
import ctypes as C
import os
import subprocess

from stitch_b200 import _abi, _lib
from stitch_b200._abi import StitchContig, StitchOpts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL_DIR = os.path.join(ROOT, "tests", "emul")
EMUL_RESULTS = {"n_reads": "emul_results_n_reads", "read": "emul_results_read", "chains": "emul_results_chains",
                "ops": "emul_results_ops", "free": "emul_free_results"}
_libs = {}


def build():
    """(Re)builds the emulator libraries when a source is newer.  On a box where that fails (the GPU box may see other
    timestamps than the container the libraries were built in) the libraries shipped with the tree are used as they are."""
    try:
        subprocess.check_call(["make", "-s", "-C", EMUL_DIR, "all"], stderr=subprocess.DEVNULL)
    except (subprocess.CalledProcessError, OSError):
        if not all(os.path.exists(os.path.join(EMUL_DIR, f"libemul_s{k}.so")) for k in (1, 2, 8)):
            raise


def lib(strip=8):
    if strip in _libs:
        return _libs[strip]
    build()
    e = C.CDLL(os.path.join(EMUL_DIR, f"libemul_s{strip}.so"))
    e.emul_create.restype = C.c_int
    e.emul_create.argtypes = [C.POINTER(StitchOpts), C.POINTER(StitchContig), C.c_uint32, C.c_int, C.POINTER(C.c_void_p)]
    for name in ("emul_align_batch", "emul_custom_batch"):
        f = getattr(e, name)
        f.restype = C.c_int
        f.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.c_uint32, C.c_void_p, C.c_uint32,
                      C.POINTER(C.c_void_p)]
    _lib.declare_results_api(e, EMUL_RESULTS)
    _lib.declare_sam_api(e, "emul_")
    e.emul_destroy.restype = None
    e.emul_destroy.argtypes = [C.c_void_p]
    e.emul_last_error.restype = C.c_char_p
    e.emul_last_error.argtypes = [C.c_void_p]
    e.emul_pk_plan.restype = C.c_int32
    e.emul_pk_plan.argtypes = [C.POINTER(StitchOpts), C.c_uint32, C.c_uint32]
    e.emul_path_counters.restype = None
    e.emul_path_counters.argtypes = [C.POINTER(C.c_ulonglong)]
    e.emul_struct_sizes.restype = None
    e.emul_struct_sizes.argtypes = [C.POINTER(C.c_uint32)]
    _libs[strip] = e
    return e


STRUCT_NAMES = ("JumpInfo", "PkRowM", "PkQuiet", "ContigEntry", "PkColConst", "RowM", "XsPart", "CmPart", "ICarry")


def struct_sizes(strip=8):
    """sizeof of the structs the kernels' shared-memory layouts are carved from: {name: bytes}."""
    out = (C.c_uint32 * len(STRUCT_NAMES))()
    lib(strip).emul_struct_sizes(out)
    return dict(zip(STRUCT_NAMES, out))


def pk_plan(opts: StitchOpts, n, m_max, strip=8):
    """pk_plan (stitch_b200/csrc/dp_packed.h) of the scoring the product derives from `opts`: the packed path's length bits,
    0 = the wide path, -1 = options the product refuses."""
    return lib(strip).emul_pk_plan(C.byref(opts), n, m_max)


def path_counters(strip=8):
    """Fills the emulator has run so far in this process: {"packed": .., "wide": .., "lb": {LB: packed fills with LB}}."""
    out = (C.c_ulonglong * 34)()
    lib(strip).emul_path_counters(out)
    return {"packed": out[0], "wide": out[1], "lb": {k: out[2 + k] for k in range(32) if out[2 + k]}}


class EmulError(RuntimeError):
    pass


class EmulAligners:
    def __init__(self, opts: StitchOpts, contigs, strip=8):
        self.e = lib(strip)
        arr, self._keep = _abi.make_contigs(contigs)
        self.n_strands = len(contigs) * (2 if opts.double_strand else 1)
        h = C.c_void_p()
        rc = self.e.emul_create(C.byref(opts), arr, len(contigs), 0, C.byref(h))
        if rc != 0:
            raise EmulError(f"create failed ({rc}): {self.e.emul_last_error(None).decode()}")
        self._h = h

    def batch(self, reads, subsets=None, raw=False):
        buf, offs = _abi.pack_reads(reads)
        words, stride = None, 0
        if subsets is not None:
            stride = (self.n_strands + 31) // 32
            words = (C.c_uint32 * (stride * len(reads)))()
            for r, sub in enumerate(subsets):
                for c in (sub or ()):
                    words[r * stride + c // 32] |= 1 << (c % 32)
        res = C.c_void_p()
        fn = self.e.emul_custom_batch if raw else self.e.emul_align_batch
        rc = fn(self._h, buf, offs, len(reads), words, stride, C.byref(res))
        if rc != 0:
            raise EmulError(f"batch failed ({rc}): {self.e.emul_last_error(self._h).decode()}")
        try:
            self.last_prealign_scores = _lib.read_prealign(self.e, "emul_", res, len(reads))
            return _lib.read_results(self.e, EMUL_RESULTS, res)
        finally:
            self.e.emul_free_results(res)

    def prealign_batch(self, reads):
        return _lib.prealign_batch(self.e, "emul_", self._h, reads, self.n_strands)

    def batch_sam(self, reads, headers, quals=None, sam_opts=None):
        """align_batch + the product's SAM record layer (host code shared with the CUDA library)."""
        buf, offs = _abi.pack_reads(reads)
        res = C.c_void_p()
        rc = self.e.emul_align_batch(self._h, buf, offs, len(reads), None, 0, C.byref(res))
        if rc != 0:
            raise EmulError(f"batch failed ({rc}): {self.e.emul_last_error(self._h).decode()}")
        try:
            chains = _lib.read_results(self.e, EMUL_RESULTS, res)
            pre = _lib.read_prealign(self.e, "emul_", res, len(reads))
            self.last_prealign_scores = pre
            sam = [_lib.format_sam(self.e, "emul_", self._h, res, r, headers[r], bytes(reads[r]),
                                   None if quals is None else quals[r], pre[r], sam_opts) for r in range(len(reads))]
            return chains, sam
        finally:
            self.e.emul_free_results(res)

    def close(self):
        if self._h:
            self.e.emul_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
