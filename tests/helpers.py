"""Shared helpers for the parity tests (test infrastructure; may import the oracle)."""
import ctypes as C
import functools
import math
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_kernels.npz")


def sample_idx(n, k=2048):
    """k distinct flat indices spread over range(n) (all of them when n <= k): a fixed stride coprime with n, no RNG, so the
    golden generator and the tests pick the same elements."""
    if n <= k:
        return np.arange(n)
    p = 7919
    while math.gcd(p, n) != 1:
        p += 2
    return np.sort((np.arange(k, dtype=np.int64) * p) % n)


@functools.lru_cache(maxsize=None)
def ref_golden():
    """Outputs of the reference's own kernels on the tests' seeded inputs (oracle/gen_golden_ref_kernels.py)."""
    return dict(np.load(REF_GOLDEN))


# Stated fp16 tolerance for q4_matmul (SURVEY.md 8c): ours accumulates exact fp16 products in fp32, so the
# only error against the float64 restatement is the final fp16 rounding (2^-11 relative) plus fp32 summation.
REL_TOL = 1.5e-3
RMS_TOL = 1.5e-3


def assert_close_ref64(got_f16, ref64, rel=REL_TOL, rms=RMS_TOL, what=""):
    got = np.asarray(got_f16, dtype=np.float64)
    ref = np.asarray(ref64, dtype=np.float64)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    assert np.isfinite(got).all(), f"{what}: non-finite output"
    r = np.sqrt(np.mean(ref * ref))
    err = np.abs(got - ref)
    bound = rel * np.abs(ref) + rms * r
    bad = err > bound
    assert not bad.any(), (f"{what}: {bad.sum()} / {bad.size} outside tolerance; max err {err.max():.4g} "
                           f"(rms ref {r:.4g}) at {np.unravel_index(err.argmax(), err.shape)}")
    return float(np.sqrt(np.mean(err * err)) / max(r, 1e-30))


def ulp_diff_f16(a, b):
    """Distance in fp16 ulps (monotone integer mapping of the bit patterns)."""
    def key(x):
        u = np.asarray(x, dtype=np.float16).view(np.uint16).astype(np.int32)
        return np.where(u & 0x8000, -(u & 0x7fff), u & 0x7fff)
    return np.abs(key(a) - key(b))


def to_cuda(*arrays):
    import torch
    out = []
    for a in arrays:
        out.append(None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda())
    return out if len(out) > 1 else out[0]


class RefLib:
    """oracle/_ref/libexllama_ref.so: the reference's own kernels compiled for sm_100a (GPU box only)."""

    def __init__(self):
        from oracle import oracle as O
        path = O.ref_cuda_lib_path()
        if path is None:
            raise FileNotFoundError("oracle/_ref/libexllama_ref.so not built")
        self.lib = C.CDLL(path)
        self.lib.ref_make_q4.restype = C.c_void_p
        self.lib.ref_make_q4.argtypes = [C.c_void_p] * 4 + [C.c_int] * 4
        self.lib.ref_q4_matmul.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        self.lib.ref_reconstruct.argtypes = [C.c_void_p, C.c_void_p]
        self.lib.ref_q4_get_x_map.argtypes = [C.c_void_p, C.c_void_p]
        self.lib.ref_prepare_buffers.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        self.lib.ref_rms_norm.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_int, C.c_int]
        self.lib.ref_rope.argtypes = [C.c_void_p] * 3 + [C.c_int] * 5
        self.lib.ref_column_remap.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        self.lib.ref_half_matmul_cublas.argtypes = [C.c_void_p] * 3 + [C.c_int] * 4
        self.lib.ref_q4_attn.argtypes = ([C.c_void_p, C.c_void_p, C.c_float] + [C.c_void_p] * 8 + [C.c_int] * 7 +
                                         [C.c_void_p, C.c_void_p, C.c_int, C.c_int])
        self.lib.ref_q4_attn_2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        self.lib.ref_q4_mlp.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        self.keep = []

    def prepare_buffers(self, inter, max_rows=2048, dq_numel=0):
        import torch
        ts = torch.zeros((max_rows, inter), dtype=torch.float16, device="cuda")
        tm = torch.zeros((4, inter), dtype=torch.float16, device="cuda")
        tz = torch.zeros((1, 65536), dtype=torch.float32, device="cuda")
        dq = torch.zeros((1, max(dq_numel, 8)), dtype=torch.float16, device="cuda")
        self.keep += [ts, tm, tz, dq]
        torch.cuda.synchronize()
        self.lib.ref_prepare_buffers(0, ts.data_ptr(), ts.numel(), tm.data_ptr(), tz.data_ptr(), dq.data_ptr(), 65536)

    def make_q4(self, qweight, qzeros, scales, g_idx_np=None):
        """qweight etc. are CUDA tensors (qweight is rewritten in place for act-order)."""
        import torch
        torch.cuda.synchronize()
        g = None
        if g_idx_np is not None:
            g = np.ascontiguousarray(g_idx_np, dtype=np.int32)
            self.keep.append(g)
        h = self.lib.ref_make_q4(qweight.data_ptr(), qzeros.data_ptr(), scales.data_ptr(),
                                 g.ctypes.data if g is not None else None,
                                 qweight.shape[0] * 8, qweight.shape[1], qzeros.shape[0], 0)
        self.keep += [qweight, qzeros, scales]
        self.lib.ref_sync()
        return h

    def q4_matmul(self, x, h, N, out=None, no_zero=False, mode=0):
        import torch
        if out is None:
            out = torch.empty((x.shape[0], N), dtype=torch.float16, device="cuda")
        torch.cuda.synchronize()
        self.lib.ref_q4_matmul(x.data_ptr(), x.shape[0], h, out.data_ptr(), int(no_zero), mode)
        self.lib.ref_sync()
        return out

    def sync(self):
        self.lib.ref_sync()
