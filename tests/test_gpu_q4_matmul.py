"""GPU parity of q4_matmul through the C ABI (ctypes -> libexl_b200.so), against the float64 oracle on the same
seeded inputs, and against the outputs of the reference's own kernels compiled for sm_100a (tests/golden/ref_kernels.npz).
Tolerance: see helpers.REL_TOL / RMS_TOL (fp16 output rounding)."""
import numpy as np
import pytest

from helpers import assert_close_ref64, ref_golden, sample_idx, to_cuda

pytestmark = pytest.mark.gpu


def _mk(oracle, K, N, gs, act, seed):
    qw, qz, sc, g_idx = oracle.synth_q4(K, N, gs, act_order=act, seed=seed)
    return qw, qz, sc, g_idx


def _q4(capi, qw, qz, sc, g_idx):
    import torch
    tq, tz, ts = to_cuda(qw.copy(), qz, sc)
    g = None if g_idx is None else torch.from_numpy(g_idx)
    return capi.Q4(tq, tz, ts, g)


SMALL = [  # (M, K, N, groupsize, act_order)
    (1, 256, 128, 128, False),
    (1, 512, 256, 32, False),
    (2, 1024, 384, 128, False),
    (3, 512, 160, 64, True),      # N not a multiple of 128
    (5, 2048, 512, 128, True),
    (7, 4096, 256, 128, False),
    (8, 1024, 1024, 1024, False),  # no groups
    (1, 11008 // 4 // 32 * 32, 128, 32, True),
    (4, 4096 + 32, 96, 32, False),  # K not a multiple of 64
]


@pytest.mark.parametrize("M,K,N,gs,act", SMALL)
def test_skinny_vs_ref64(oracle, M, K, N, gs, act):
    import torch
    from exllama_b200 import capi
    qw, qz, sc, g_idx = _mk(oracle, K, N, gs, act, seed=K + N + M)
    x = oracle.synth_x(M, K, seed=M)
    q4 = _q4(capi, qw, qz, sc, g_idx)
    out = capi.q4_matmul(to_cuda(x), q4, force_path=1)
    torch.cuda.synchronize()
    assert capi.last_q4_path() == "skinny_mma"
    ref = oracle.ref64_with_act_order(x, qw, qz, sc, g_idx)
    assert_close_ref64(out.cpu().numpy(), ref, what=f"skinny M{M} K{K} N{N} g{gs} act{act}")
    if act:
        # make_q4 contract: x_map equals the oracle's, caller's qweight rewritten in place (q4_matrix.cu:159)
        xm = oracle.make_x_map(g_idx, K // gs)
        np.testing.assert_array_equal(q4.x_map(), xm)
        np.testing.assert_array_equal(q4.qweight.cpu().numpy(), oracle.make_sequential(qw, xm))


@pytest.mark.parametrize("M,K,N,gs,act", [(2, 1024, 384, 128, False), (6, 2048, 512, 32, True)])
def test_skinny_accumulate(oracle, M, K, N, gs, act):
    """no_zero: out += x.W  (residual add of q4_attn_2 / q4_mlp, q4_matmul.cu:78-82)"""
    import torch
    from exllama_b200 import capi
    qw, qz, sc, g_idx = _mk(oracle, K, N, gs, act, seed=11)
    x = oracle.synth_x(M, K, seed=3)
    res = oracle.synth_x(M, N, seed=4)
    q4 = _q4(capi, qw, qz, sc, g_idx)
    out = to_cuda(res.copy())
    capi.q4_matmul(to_cuda(x), q4, out=out, no_zero=True, force_path=1)
    ref = oracle.ref64_with_act_order(x, qw, qz, sc, g_idx, acc_in=res)
    assert_close_ref64(out.cpu().numpy(), ref, what="accumulate")


def test_deterministic(oracle):
    """stream-K fix-up sums partials in a fixed order: bitwise identical across launches (the reference's
    fp16 atomics are not, q4_matmul.cu:203-211)."""
    import torch
    from exllama_b200 import capi
    qw, qz, sc, _ = _mk(oracle, 4096, 4096, 128, False, seed=1)
    x = to_cuda(oracle.synth_x(3, 4096))
    q4 = _q4(capi, qw, qz, sc, None)
    a = capi.q4_matmul(x, q4).clone()
    for _ in range(5):
        b = capi.q4_matmul(x, q4)
        assert torch.equal(a, b)


def test_full_size_7b_shapes_linearity(oracle):
    """BASELINE-size shapes: the oracle is too slow at full size, so check size-independent properties:
    (a) linearity in x: W(x1 + x2) == W x1 + W x2 within fp16 tolerance,
    (b) a sampled set of output columns against ref64 (column sub-matrix is an exact restriction)."""
    import torch
    from exllama_b200 import capi
    for (K, N, gs) in [(4096, 4096, 128), (4096, 11008, 128), (11008, 4096, 128)]:
        qw, qz, sc, _ = _mk(oracle, K, N, gs, False, seed=K + N)
        q4 = _q4(capi, qw, qz, sc, None)
        x1 = oracle.synth_x(1, K, seed=1); x2 = oracle.synth_x(1, K, seed=2)
        xs = (x1.astype(np.float32) + x2.astype(np.float32)).astype(np.float16)
        y1 = capi.q4_matmul(to_cuda(x1), q4).float(); y2 = capi.q4_matmul(to_cuda(x2), q4).float()
        ys = capi.q4_matmul(to_cuda(xs), q4).float()
        # xs was rounded to fp16: compare against W applied to the rounded sum via the column sample instead
        cols = np.sort(np.random.default_rng(0).choice(N // 8, 24, replace=False)) * 8
        cols = (cols[:, None] + np.arange(8)[None]).reshape(-1)
        sub_qw = np.ascontiguousarray(qw[:, cols]); sub_sc = np.ascontiguousarray(sc[:, cols])
        zfull = ((qz.view(np.uint32)[:, :, None] >> (np.arange(8, dtype=np.uint32) * 4)[None, None]) & 0xF).reshape(K // gs, N)
        zsub = zfull[:, cols].reshape(K // gs, -1, 8)
        sub_qz = (zsub.astype(np.uint32) << (np.arange(8, dtype=np.uint32) * 4)).sum(-1).astype(np.uint32).view(np.int32)
        for xv, yv in ((x1, y1), (x2, y2), (xs, ys)):
            ref = oracle.q4_matmul_f64(xv, sub_qw, sub_qz, sub_sc)
            assert_close_ref64(yv.cpu().numpy()[:, cols], ref, what=f"col-sample K{K} N{N}")
        rms = float(ys.pow(2).mean().sqrt())
        assert float((y1 + y2 - ys).abs().max()) <= 0.02 * rms + 4e-3 * float(ys.abs().max())


@pytest.mark.parametrize("M", [9, 17, 64])
def test_mid_m_route(oracle, M):
    """8 < M <= 64 takes repeated skinny passes (HBM-bound regime) -- same results as the oracle."""
    from exllama_b200 import capi
    K, N, gs = 1024, 512, 128
    qw, qz, sc, g_idx = _mk(oracle, K, N, gs, True, seed=9)
    x = oracle.synth_x(M, K, seed=5)
    q4 = _q4(capi, qw, qz, sc, g_idx)
    out = capi.q4_matmul(to_cuda(x), q4)
    assert_close_ref64(out.cpu().numpy(), oracle.ref64_with_act_order(x, qw, qz, sc, g_idx), what=f"mid M={M}")


@pytest.mark.parametrize("M,K,N,gs,act", [(128, 1024, 512, 128, False), (200, 2048, 384, 32, True)])
def test_recons_cublas_path(oracle, M, K, N, gs, act):
    """force_path=3: reconstruct + cuBLAS (the reference's own prefill algorithm, q4_matmul.cu:301-344)."""
    from exllama_b200 import capi
    qw, qz, sc, g_idx = _mk(oracle, K, N, gs, act, seed=21)
    x = oracle.synth_x(M, K, seed=6)
    q4 = _q4(capi, qw, qz, sc, g_idx)
    out = capi.q4_matmul(to_cuda(x), q4, force_path=3)
    assert capi.last_q4_path() == "recons_cublas"
    ref = oracle.ref64_with_act_order(x, qw, qz, sc, g_idx, recons=True)
    assert_close_ref64(out.cpu().numpy(), ref, what="recons")


@pytest.mark.parametrize("M,K,N,gs,act", [(1, 768, 256, 96, False), (5, 1152, 160, 192, True)])
def test_skinny_unsupported_groupsize_takes_general_route(oracle, M, K, N, gs, act):
    """A group size that is not 32 * 2^n cannot go through the skinny kernel; instead of an error (ADVICE r1) the call takes the
    reconstruct + cuBLAS route, which handles any GPTQ shape the reference's kernels handle."""
    from exllama_b200 import capi
    qw, qz, sc, g_idx = _mk(oracle, K, N, gs, act, seed=33)
    x = oracle.synth_x(M, K, seed=8)
    q4 = _q4(capi, qw, qz, sc, g_idx)
    out = capi.q4_matmul(to_cuda(x), q4)
    assert capi.last_q4_path() == "recons_cublas"
    ref = oracle.ref64_with_act_order(x, qw, qz, sc, g_idx, recons=True)
    assert_close_ref64(out.cpu().numpy(), ref, what=f"general route gs={gs}")


TC_CASES = [(128, 1024, 512, 128, False), (200, 2048, 384, 32, True), (1, 512, 128, 64, False), (77, 4096, 1152, 128, True),
            (384, 1024, 1024, 1024, False), (130, 2816, 96, 128, False)]


@pytest.mark.parametrize("M,K,N,gs,act", TC_CASES)
def test_tcgen05_gemm_vs_ref64(oracle, M, K, N, gs, act):
    """force_path=2: the tcgen05 fused-dequant GEMM.  Its B operand is bit-identical to the reference's reconstructed
    weights (fp16-rounded scale * (q - zp)), accumulated in fp32 -> compare against the `recons` flavour of ref64."""
    import torch
    from exllama_b200 import capi
    qw, qz, sc, g_idx = _mk(oracle, K, N, gs, act, seed=K + N + M)
    x = oracle.synth_x(M, K, seed=M)
    q4 = _q4(capi, qw, qz, sc, g_idx)
    out = capi.q4_matmul(to_cuda(x), q4, force_path=2)
    torch.cuda.synchronize()
    assert capi.last_q4_path() == "tc_gemm"
    ref = oracle.ref64_with_act_order(x, qw, qz, sc, g_idx, recons=True)
    assert_close_ref64(out.cpu().numpy(), ref, what=f"tc_gemm M{M} K{K} N{N} g{gs} act{act}")
    res = oracle.synth_x(M, N, seed=99)
    out2 = to_cuda(res.copy())
    capi.q4_matmul(to_cuda(x), q4, out=out2, no_zero=True, force_path=2)
    ref2 = oracle.ref64_with_act_order(x, qw, qz, sc, g_idx, acc_in=res, recons=True)
    assert_close_ref64(out2.cpu().numpy(), ref2, what="tc_gemm accumulate")


def test_reconstruct_bit_exact(oracle):
    from exllama_b200 import capi
    for (K, N, gs) in [(256, 64, 32), (1024, 384, 128)]:
        qw, qz, sc, _ = _mk(oracle, K, N, gs, False, seed=31)
        q4 = _q4(capi, qw, qz, sc, None)
        got = capi.q4_reconstruct(q4).cpu().numpy()
        np.testing.assert_array_equal(got.view(np.uint16), oracle.reconstruct_f16(qw, qz, sc).view(np.uint16))


# ---------------------------------------------------------------------------------------------------
# against the reference's own kernels (outputs stored by oracle/gen_golden_ref_kernels.py)
# ---------------------------------------------------------------------------------------------------

REF_DECODE_CASES = [(1, 4096, 4096, 128, False), (1, 4096, 11008, 128, False), (4, 5120, 5120, 128, True), (7, 2048, 6656, 32, True)]
REF_RECONS_CASE = (64, 4096, 4096, 128)


def ref_decode_inputs(oracle, M, K, N, gs, act):
    return _mk(oracle, K, N, gs, act, seed=41) + (oracle.synth_x(M, K, seed=7),)


def ref_recons_inputs(oracle):
    M, K, N, gs = REF_RECONS_CASE
    return _mk(oracle, K, N, gs, False, seed=43)[:3] + (oracle.synth_x(M, K, seed=8),)


@pytest.mark.parametrize("M,K,N,gs,act", REF_DECODE_CASES)
def test_against_reference_decode_kernel(oracle, M, K, N, gs, act):
    """|new - ref_ext| within 2e-2 (the reference accumulates in fp16 with atomics) AND our error against the
    float64 restatement is no larger than the reference's own (SURVEY.md 8c).  Compared at helpers.sample_idx positions."""
    from exllama_b200 import capi
    qw, qz, sc, g_idx, x = ref_decode_inputs(oracle, M, K, N, gs, act)
    g = ref_golden()
    key = f"q4_decode_{M}_{K}_{N}_{gs}_{int(act)}"
    idx = sample_idx(M * N)
    mine = capi.q4_matmul(to_cuda(x), _q4(capi, qw, qz, sc, g_idx)).cpu().numpy().astype(np.float64).reshape(-1)[idx]
    theirs = g[key].astype(np.float64)
    if act:
        # both implementations must have produced the same sequential qweight and x_map
        seq = oracle.make_sequential(qw, oracle.make_x_map(g_idx, K // gs)).reshape(-1)
        np.testing.assert_array_equal(g[key + "_qweight"], seq[sample_idx(seq.size)])
    # column sample for ref64 (full oracle is O(MKN) on the CPU)
    ref_full = oracle.ref64_with_act_order(x, qw, qz, sc, g_idx).reshape(-1)[idx] if K * N <= 4096 * 4096 * 2 else None
    rms = np.sqrt(np.mean(theirs ** 2))
    assert np.all(np.abs(mine - theirs) <= 2e-2 * np.abs(theirs) + 2e-2 * rms)
    if ref_full is not None:
        e_mine = np.sqrt(np.mean((mine - ref_full) ** 2)); e_ref = np.sqrt(np.mean((theirs - ref_full) ** 2))
        assert e_mine <= e_ref * 1.05 + 1e-6, (e_mine, e_ref)


def test_against_reference_recons_path(oracle):
    from exllama_b200 import capi
    qw, qz, sc, x = ref_recons_inputs(oracle)
    out = capi.q4_matmul(to_cuda(x), _q4(capi, qw, qz, sc, None)).cpu().numpy().astype(np.float64).reshape(-1)
    mine = out[sample_idx(out.size)]
    theirs = ref_golden()["q4_recons"].astype(np.float64)
    rms = np.sqrt(np.mean(theirs ** 2))
    assert np.all(np.abs(mine - theirs) <= 2e-2 * np.abs(theirs) + 2e-2 * rms)
