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


def rms(a):
    return float(np.sqrt(np.mean(np.square(np.asarray(a, dtype=np.float64)))))


def sharper(fused, per_op, want, what):
    """fused-vs-oracle rms error <= 1.25 x per-op-vs-oracle rms error + 1e-4 x rms; returns the ratio of the two errors.
    Both paths round to fp16 at the same points, so a defect of the fused path alone shows up here long before it reaches an
    elementwise tolerance.  Outputs one fp16 rounding from the oracle on both paths (errors ~1e-4 of rms), where single-ulp
    rounding flips alone move the ratio up to ~1.5 (measured on a B200, median 0.98 over all decode-step cases): the
    1e-4 x rms term covers that."""
    want = np.asarray(want, dtype=np.float64).reshape(-1)
    e_f = rms(np.asarray(fused, dtype=np.float64).reshape(-1) - want)
    e_p = rms(np.asarray(per_op, dtype=np.float64).reshape(-1) - want)
    r = rms(want)
    assert e_f <= 1.25 * e_p + 1e-4 * r, f"{what}: fused rms err {e_f:.4g} vs per-op {e_p:.4g} (rms {r:.4g})"
    ratio = e_f / max(e_p, 1e-30)
    print(f"{what}: fused/per-op rms error ratio {ratio:.3f} (fused {e_f / r:.3e}, per-op {e_p / r:.3e} of rms)")
    return ratio


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


# ---------------------------------------------------------------------------------------------------
# large GEMMs: float64 reference on a row / column sample
# ---------------------------------------------------------------------------------------------------

def tile_edge_sample(n, tile=128, edge=8):
    """Sorted indices of range(n): the first and last `edge` of every full `tile`-sized block, and all of a partial last block
    (where the tail handling of a tiled kernel lives)."""
    full = n // tile
    idx = [np.arange(b * tile, b * tile + edge) for b in range(full)] + [np.arange((b + 1) * tile - edge, (b + 1) * tile) for b in range(full)]
    idx.append(np.arange(full * tile, n))
    return np.unique(np.concatenate(idx)).astype(np.int64)


def ref64_sampled(x, qw, qz, sc, g_idx, rows, cols, acc_in=None, recons=True):
    """ref64_with_act_order(...)[rows][:, cols] without the full M x K x N contraction.  Both restrictions are exact: a row of the
    product depends on that row of x only, a column on that column of the GPTQ tensors (and on g_idx, a property of K).
    cols must be a multiple of 8 long (the zero points are repacked 8 per word)."""
    from exllama_b200.tp import gather_q4_columns
    from oracle import oracle as O
    rows, cols = np.asarray(rows), np.asarray(cols)
    xm = None
    if g_idx is not None:
        xm = O.make_x_map(g_idx, qz.shape[0])
        qw = O.make_sequential(qw, xm)
    sqw, sqz, ssc = gather_q4_columns(qw, qz, sc, cols)
    acc = None if acc_in is None else np.ascontiguousarray(acc_in[rows][:, cols])
    return O.q4_matmul_f64(np.ascontiguousarray(x[rows]), sqw, sqz, ssc, xm, acc, recons)


# ---------------------------------------------------------------------------------------------------
# decode step: synthetic stack and its float64 / fp16 oracle composition
# ---------------------------------------------------------------------------------------------------

def mk_stack(hidden, inter, layers, heads, gs, max_seq, vocab=2048, seed=3, act=False, with_head=True):
    """Seeded synthetic GPTQ stack on cuda:0 with random (not zero) KV caches."""
    import torch
    from exllama_b200.stack import DecodeStack, LlamaShape
    shape = LlamaShape("synthetic", hidden, inter, layers, heads, vocab=vocab)
    st = DecodeStack(shape, groupsize=gs, act_order=act, device="cuda:0", max_seq=max_seq, seed=seed, with_head=with_head)
    g = torch.Generator(device="cuda"); g.manual_seed(seed + 100)
    for kc, vc in zip(st.key_cache, st.value_cache):
        kc.copy_((torch.randn(kc.shape, device="cuda", generator=g) * 0.5).half())
        vc.copy_((torch.randn(vc.shape, device="cuda", generator=g) * 0.5).half())
    return st


def oracle_step(oracle, st, x, past):
    """float64/fp16 restatement of one decode token through the stack: returns (final hidden fp16, logits float64 or None without
    lm_head, new k/v rows)."""
    s = st.shape
    hd, heads = s.head_dim, s.heads
    sin = st.sin.view(-1, hd).cpu().numpy(); cos = st.cos.view(-1, hd).cpu().numpy()
    x = x.reshape(1, s.hidden).copy()
    rows = []

    def mm(xin, lin, acc=None):
        # make_q4 has already rewritten an act-order qweight into sequential order (q4_matrix.cu:159): contract with the x gather
        xm = None if lin.g_idx is None else oracle.make_x_map(lin.g_idx.numpy(), lin.qzeros.shape[0])
        return oracle.q4_matmul_f64(xin, lin.qweight.cpu().numpy(), lin.qzeros.cpu().numpy(), lin.scales.cpu().numpy(), xm, acc)
    for i, L in enumerate(st.layers):
        xn, _ = oracle.rms_norm(x, L.ln1.cpu().numpy(), s.eps)
        q = mm(xn, L.q).astype(np.float16); k = mm(xn, L.k).astype(np.float16); v = mm(xn, L.v).astype(np.float16)
        q = oracle.rope(q.reshape(1, heads, hd), sin, cos, 1, heads, hd, heads, past).reshape(-1)
        k = oracle.rope(k.reshape(1, heads, hd), sin, cos, 1, heads, hd, heads, past).reshape(heads, hd)
        kc = st.key_cache[i][0].cpu().numpy().copy(); vc = st.value_cache[i][0].cpu().numpy().copy()
        kc[:, past] = k; vc[:, past] = v.reshape(heads, hd)
        rows.append((k.copy(), v.reshape(heads, hd).copy()))
        attn = oracle.decode_attn_f64(q, kc, vc, heads, heads, hd, past + 1, st.max_seq).astype(np.float16).reshape(1, -1)
        x = mm(attn, L.o, acc=x).astype(np.float16)
        xn, _ = oracle.rms_norm(x, L.ln2.cpu().numpy(), s.eps)
        act = oracle.silu_mul(mm(xn, L.gate).astype(np.float16), mm(xn, L.up).astype(np.float16))
        x = mm(act, L.down, acc=x).astype(np.float16)
    if st.lm_head is None:
        return x, None, rows
    hn, _ = oracle.rms_norm(x, st.norm.cpu().numpy(), s.eps)
    hn = hn.astype(np.float64).reshape(-1)
    # in row blocks: a 32000 x 8192 head in float64 alone would be 2 GB of host memory
    logits = np.concatenate([st.lm_head[r:r + 4096].cpu().numpy().astype(np.float64) @ hn for r in range(0, s.vocab, 4096)])
    return x, logits.reshape(1, -1), rows
