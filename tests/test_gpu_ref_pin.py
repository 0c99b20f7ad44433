"""Pins the oracle AND this repo's kernels against the reference's OWN kernels for every op of SURVEY.md 8a that the
q4_matmul tests do not already cover (VERDICT r1 "What's weak" 1a): rms_norm, rope, column_remap, half_matmul_cublas and
the fused decoder blocks q4_attn / q4_attn_2 / q4_mlp (which contain update_cache and silu_mul).

Three-way comparison on the same seeded inputs:
    reference kernel (its outputs stored in tests/golden/ref_kernels.npz by oracle/gen_golden_ref_kernels.py, which runs
                      oracle/_ref/libexllama_ref.so: the reference's sources compiled for sm_100a)
    oracle           (oracle/gptq_oracle.c, CPU restatement)
    ours             (libexl_b200.so through the C ABI)
Outputs larger than 2048 elements are compared at the helpers.sample_idx positions the fixture stores.
Bit-exact where the arithmetic is elementwise fp16 (rope, column_remap, cache rows); a stated tolerance where the
reference itself is not reproducible (fp32 atomics in rms_norm: <= 2 fp16 ulp; fp16 atomics in q4_matmul: 2e-2).

Also: full-size parity of every SURVEY.md 8d shape (13B act-order, 33B g32 act-order, 65B) at M in {1, 4, 7}, column
sampled against ref64, and the reference's own run-to-run spread (SURVEY.md 8c) against ours.
"""
import json
import os

import numpy as np
import pytest

from helpers import ROOT, assert_close_ref64, ref_golden, sample_idx, to_cuda, ulp_diff_f16

pytestmark = pytest.mark.gpu

RMS_CASES = [(1, 4096), (1, 5120), (3, 6656), (7, 8192), (17, 4096)]
ROPE_CASES = [(1, 1, 32, 128, 0), (1, 1, 40, 128, 1919), (1, 5, 8, 128, 3), (2, 3, 4, 128, 100)]
ATTN_CASES = [(1, 0), (1, 37), (2, 5)]          # (q_len, past) of q4_attn
BLOCK_ROWS = [1, 2]                              # rows of q4_attn_2 / q4_mlp
ATTN_SHAPE = dict(hidden=1024, heads=8, hd=128, gs=128, max_seq=64)
MLP_SHAPE = dict(hidden=1024, inter=2816, gs=128)
SPREAD_SHAPE = (4096, 4096, 128)


def _sincos(max_seq, hd):
    inv = 1.0 / (10000 ** (np.arange(0, hd, 2, dtype=np.float64) / hd))
    ang = np.outer(np.arange(max_seq), inv)
    emb = np.concatenate([ang, ang], -1)
    return np.sin(emb).astype(np.float16), np.cos(emb).astype(np.float16)


def _flat(a, idx=None):
    a = np.asarray(a).reshape(-1)
    return a[sample_idx(a.size) if idx is None else idx]


# ---- seeded inputs (oracle/gen_golden_ref_kernels.py runs the reference on exactly these) --------------------------------

def rms_norm_inputs(rows, dim):
    rng = np.random.default_rng(rows * 31 + dim)
    x = rng.standard_normal((rows, dim)).astype(np.float16)
    w = (1 + 0.1 * rng.standard_normal(dim)).astype(np.float16)
    return x, w


def rope_inputs(bsz, q_len, heads, hd, past):
    rng = np.random.default_rng(17 + past)
    x = rng.standard_normal((bsz, q_len, heads * hd)).astype(np.float16)
    sin, cos = _sincos(2048, hd)
    return x, sin, cos


def column_remap_inputs():
    rng = np.random.default_rng(3)
    out = []
    for M, K in ((1, 4096), (7, 5120), (33, 6656)):
        x = rng.standard_normal((M, K)).astype(np.float16)
        out.append((x, rng.permutation(K).astype(np.uint32)))
    return out


def half_matmul_inputs():
    rng = np.random.default_rng(4)
    out = []
    for M, K, N in ((1, 4096, 16), (5, 512, 64), (16, 64, 4096)):
        x = rng.standard_normal((M, K)).astype(np.float16)
        out.append((x, (rng.standard_normal((K, N)) * 0.1).astype(np.float16)))
    return out


def _layer(oracle, hidden, inter, gs, act, seed):
    names = [("q", hidden, hidden), ("k", hidden, hidden), ("v", hidden, hidden), ("o", hidden, hidden),
             ("gate", hidden, inter), ("up", hidden, inter), ("down", inter, hidden)]
    return {n: oracle.synth_q4(K, N, gs, act_order=act, seed=seed + i) for i, (n, K, N) in enumerate(names)}


def q4_attn_inputs(oracle, act, q_len):
    s = ATTN_SHAPE
    t = _layer(oracle, s["hidden"], 2048, s["gs"], act, seed=300)
    rng = np.random.default_rng(11)
    x = rng.standard_normal((1, q_len, s["hidden"])).astype(np.float16)
    w = (1 + 0.1 * rng.standard_normal(s["hidden"])).astype(np.float16)
    sin, cos = _sincos(s["max_seq"], s["hd"])
    return t, x, w, sin, cos


def block_inputs(oracle, act, rows):
    s = MLP_SHAPE
    t = _layer(oracle, s["hidden"], s["inter"], s["gs"], act, seed=400)
    rng = np.random.default_rng(12)
    x = rng.standard_normal((rows, s["hidden"])).astype(np.float16)
    attn = rng.standard_normal((rows, s["hidden"])).astype(np.float16)
    w = (1 + 0.1 * rng.standard_normal(s["hidden"])).astype(np.float16)
    return t, x, attn, w


def spread_inputs(oracle):
    K, N, gs = SPREAD_SHAPE
    qw, qz, sc, _ = oracle.synth_q4(K, N, gs, seed=5)
    return qw, qz, sc, oracle.synth_x(1, K, seed=6)


# ---- tests --------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("rows,dim", RMS_CASES)
def test_rms_norm_three_way(oracle, rows, dim):
    from exllama_b200 import capi
    x, w = rms_norm_inputs(rows, dim)
    want, _ = oracle.rms_norm(x, w, 1e-6)
    ref = ref_golden()[f"rms_norm_{rows}_{dim}"]
    mine = _flat(capi.rms_norm(*to_cuda(x, w), 1e-6).cpu().numpy())
    # the reference sums x^2 with float atomics (rms_norm.cu:20-79): its row factor can move by one fp16 ulp run to run
    assert ulp_diff_f16(ref, _flat(want)).max() <= 2, "oracle rms_norm is not the reference's rms_norm"
    assert ulp_diff_f16(mine, ref).max() <= 2
    assert (ulp_diff_f16(mine, ref) == 0).mean() > 0.5


@pytest.mark.parametrize("bsz,q_len,heads,hd,past", ROPE_CASES)
def test_rope_three_way_bit_exact(oracle, bsz, q_len, heads, hd, past):
    from exllama_b200 import capi
    x, sin, cos = rope_inputs(bsz, q_len, heads, hd, past)
    want = oracle.rope(x.reshape(bsz, q_len * heads, hd), sin, cos, bsz, q_len * heads, hd, heads, past).reshape(x.shape)
    ref = ref_golden()[f"rope_{bsz}_{q_len}_{heads}_{hd}_{past}"]
    tmine = to_cuda(x.copy())
    capi.rope_(tmine, *to_cuda(sin, cos), past, heads, hd)
    np.testing.assert_array_equal(ref.view(np.uint16), _flat(want).view(np.uint16), err_msg="oracle rope != reference rope")
    np.testing.assert_array_equal(tmine.cpu().numpy().view(np.uint16), want.view(np.uint16))


def test_column_remap_three_way(oracle):
    import torch
    from exllama_b200 import capi
    g = ref_golden()
    for i, (x, perm) in enumerate(column_remap_inputs()):
        want = oracle.column_remap(x, perm)
        np.testing.assert_array_equal(g[f"column_remap_{i}"], _flat(want))
        mine = capi.column_remap(to_cuda(x), torch.from_numpy(perm.view(np.int32)).cuda()).cpu().numpy()
        np.testing.assert_array_equal(mine, want)


def test_half_matmul_cublas_three_way(oracle):
    from exllama_b200 import capi
    g = ref_golden()
    for i, (x, w) in enumerate(half_matmul_inputs()):
        ref64 = oracle.half_matmul_f64(x, w)
        ref = g[f"half_matmul_cublas_{i}"]
        # the reference's Hgemm accumulates in fp16 (CUBLAS_COMPUTE_16F): looser than ours against float64
        assert_close_ref64(ref, _flat(ref64), rel=2e-2, rms=2e-2, what="reference Hgemm vs oracle")
        mine = capi.half_matmul_cublas(*to_cuda(x, w)).cpu().numpy()
        assert_close_ref64(mine, ref64, what="ours vs oracle")
        e_mine = np.abs(_flat(mine) - _flat(ref64)).max(); e_ref = np.abs(ref - _flat(ref64)).max()
        assert e_mine <= e_ref * 1.05 + 1e-4


def _close_to_reference(mine, ref, what):
    mine = np.asarray(mine, np.float64); ref = np.asarray(ref, np.float64)
    rms = np.sqrt(np.mean(ref ** 2))
    bad = np.abs(mine - ref) > 2e-2 * np.abs(ref) + 2e-2 * rms
    assert not bad.any(), f"{what}: {bad.sum()} / {bad.size} outside 2e-2 of the reference kernel; max {np.abs(mine - ref).max():.4g}, rms {rms:.4g}"


def _q4(capi, t):
    import torch
    qw, qz, sc, g = t
    return capi.Q4(*to_cuda(qw.copy(), qz, sc), None if g is None else torch.from_numpy(g))


@pytest.mark.parametrize("act", [False, True])
@pytest.mark.parametrize("q_len,past", ATTN_CASES)
def test_q4_attn_vs_reference_block(oracle, act, q_len, past):
    """ref_q4_attn (q4_attn.cu:74-165: norm -> q,k,v -> rope -> cache) next to exl_q4_attn and the oracle composition.
    The generator checked the reference's own cache layout (rows past..past+q_len hold its k / v, the rest untouched) and
    that it leaves x unmodified; here the same holds for ours."""
    import torch
    from exllama_b200 import capi
    s = ATTN_SHAPE
    hidden, heads, hd, max_seq = s["hidden"], s["heads"], s["hd"], s["max_seq"]
    t, x, w, sin, cos = q4_attn_inputs(oracle, act, q_len)
    ts, tc, tw = to_cuda(sin, cos, w)
    Q, K, V = (_q4(capi, t[n]) for n in ("q", "k", "v"))
    tx = to_cuda(x.copy())
    q = torch.zeros((1, q_len, hidden), dtype=torch.float16, device="cuda"); k = torch.zeros_like(q); v = torch.zeros_like(q)
    kc = torch.zeros((1, heads, max_seq, hd), dtype=torch.float16, device="cuda"); vc = torch.zeros_like(kc)
    capi.q4_attn(tx, tw, 1e-6, q, k, v, Q, K, V, ts, tc, q_len, past, heads, heads, hd, kc, vc, max_seq)
    torch.cuda.synchronize()
    q, k, v, kc, vc, xo = (a.cpu().numpy() for a in (q, k, v, kc, vc, tx))
    g = ref_golden()
    key = f"q4_attn_{int(act)}_{q_len}_{past}"
    for name, mine in (("q", q), ("k", k), ("v", v)):          # the caches are compared row by row below (mostly zeros: no meaningful rms)
        _close_to_reference(mine, g[f"{key}_{name}"], f"q4_attn {name}")
    np.testing.assert_array_equal(xo, x)            # x itself is not modified by q4_attn
    # cache layout: rows past..past+q_len hold k / v exactly, everything else untouched
    for tt in range(q_len):
        np.testing.assert_array_equal(kc[0, :, past + tt], k.reshape(q_len, heads, hd)[tt])
        np.testing.assert_array_equal(vc[0, :, past + tt], v.reshape(q_len, heads, hd)[tt])
    mask = np.ones(max_seq, bool); mask[past:past + q_len] = False
    assert not kc[0][:, mask].any() and not vc[0][:, mask].any()
    # the oracle composition pins the same block: v is a plain projection of the normalised x
    ref_v = g[f"{key}_v"].reshape(q_len, hidden)
    xn, _ = oracle.rms_norm(x.reshape(q_len, hidden), w, 1e-6)
    v64 = oracle.ref64_with_act_order(xn, *t["v"])
    _close_to_reference(v64, ref_v, "oracle v vs reference")
    e_mine = np.sqrt(np.mean((v.reshape(q_len, hidden) - v64) ** 2))
    e_ref = np.sqrt(np.mean((ref_v - v64) ** 2))
    assert e_mine <= e_ref * 1.05 + 1e-6, (e_mine, e_ref)


@pytest.mark.parametrize("act", [False, True])
@pytest.mark.parametrize("rows", BLOCK_ROWS)
def test_q4_attn_2_and_mlp_vs_reference_block(oracle, act, rows):
    """ref_q4_attn_2 (q4_attn.cu:206-228) and ref_q4_mlp (q4_mlp.cu:100-199) next to ours."""
    from exllama_b200 import capi
    t, x, attn, w = block_inputs(oracle, act, rows)
    g = ref_golden()
    key = f"block_{int(act)}_{rows}"

    x_ours = to_cuda(x.copy()); capi.q4_attn_2(x_ours, to_cuda(attn), _q4(capi, t["o"]))
    x_ref = g[f"{key}_attn_2"]
    want = oracle.ref64_with_act_order(attn, *t["o"], acc_in=x)
    _close_to_reference(x_ours.cpu().numpy(), x_ref, "q4_attn_2")
    _close_to_reference(want, x_ref, "oracle attn_2 vs reference")
    assert_close_ref64(x_ours.cpu().numpy(), want, what="attn_2 vs oracle")

    x_ours = to_cuda(x.copy()); capi.q4_mlp(x_ours, to_cuda(w), 1e-6, *(_q4(capi, t[n]) for n in ("gate", "up", "down")))
    xn, _ = oracle.rms_norm(x, w, 1e-6)
    g16 = oracle.ref64_with_act_order(xn, *t["gate"]).astype(np.float16)
    u16 = oracle.ref64_with_act_order(xn, *t["up"]).astype(np.float16)
    want = oracle.ref64_with_act_order(oracle.silu_mul(g16, u16), *t["down"], acc_in=x)
    # three fp16-accumulated matmuls in a row: the reference block is itself ~1e-2 from float64
    mine, ref = x_ours.cpu().numpy().astype(np.float64), g[f"{key}_mlp"].astype(np.float64)
    rms = np.sqrt(np.mean(want ** 2))
    assert np.all(np.abs(mine - ref) <= 4e-2 * np.abs(ref) + 4e-2 * rms), "q4_mlp vs reference block"
    assert np.all(np.abs(want - ref) <= 4e-2 * np.abs(ref) + 4e-2 * rms), "oracle mlp vs reference block"
    assert np.sqrt(np.mean((mine - want) ** 2)) <= np.sqrt(np.mean((ref - want) ** 2)) * 1.05 + 1e-6
# ---------------------------------------------------------------------------------------------------------
# full BASELINE sizes (SURVEY.md 8d): column-sampled ref64, M in {1, 4, 7}
# ---------------------------------------------------------------------------------------------------------

def _col_sample(qw, qz, sc, ncols8, seed=0):
    K8, N = qw.shape
    G = qz.shape[0]
    c8 = np.sort(np.random.default_rng(seed).choice(N // 8, ncols8, replace=False))
    cols = (c8[:, None] * 8 + np.arange(8)[None]).reshape(-1)
    sub_qw = np.ascontiguousarray(qw[:, cols]); sub_sc = np.ascontiguousarray(sc[:, cols])
    sub_qz = np.ascontiguousarray(qz[:, c8])          # one packed word of qzeros covers exactly 8 adjacent columns
    return cols, sub_qw, sub_qz, sub_sc


FULL = [  # (K, N, groupsize, act_order) -- every 8d shape not already covered by test_full_size_7b_shapes_linearity
    (5120, 5120, 128, True), (5120, 13824, 128, True), (13824, 5120, 128, True),
    (6656, 6656, 32, True), (6656, 17920, 32, True), (17920, 6656, 32, True),
    (8192, 8192, 128, False), (8192, 22016, 128, False), (22016, 8192, 128, False),
]


@pytest.mark.parametrize("K,N,gs,act", FULL)
def test_full_size_baseline_shapes(oracle, K, N, gs, act):
    import torch
    from exllama_b200 import capi
    qw, qz, sc, g_idx = oracle.synth_q4(K, N, gs, act_order=act, seed=K + N)
    tq, tz, ts = to_cuda(qw.copy(), qz, sc)
    q4 = capi.Q4(tq, tz, ts, None if g_idx is None else torch.from_numpy(g_idx))
    x_map = None
    qseq = qw
    if act:
        x_map = oracle.make_x_map(g_idx, K // gs)
        qseq = oracle.make_sequential(qw, x_map)
        np.testing.assert_array_equal(q4.x_map(), x_map)
    cols, sub_qw, sub_qz, sub_sc = _col_sample(qseq, qz, sc, 12, seed=N)
    for M in (1, 4, 7):
        x = oracle.synth_x(M, K, seed=M)
        out = capi.q4_matmul(to_cuda(x), q4)
        torch.cuda.synchronize()
        assert capi.last_q4_path() == "skinny_mma"
        ref = oracle.q4_matmul_f64(x, sub_qw, sub_qz, sub_sc, x_map)
        assert_close_ref64(out.cpu().numpy()[:, cols], ref, what=f"full-size K{K} N{N} g{gs} act{act} M{M}")
        res = oracle.synth_x(M, N, seed=50 + M)
        out2 = to_cuda(res.copy())
        capi.q4_matmul(to_cuda(x), q4, out=out2, no_zero=True)
        ref2 = oracle.q4_matmul_f64(x, sub_qw, sub_qz, sub_sc, x_map, acc_in=np.ascontiguousarray(res[:, cols]))
        assert_close_ref64(out2.cpu().numpy()[:, cols], ref2, what=f"full-size accumulate K{K} N{N} M{M}")



def test_reference_run_to_run_spread(oracle):
    """SURVEY.md 8c: the reference's decode kernel uses fp16 atomicAdd over K slices (q4_matmul.cu:203-211), so its
    result is not reproducible; ours is bitwise reproducible.  Three runs of each (the reference's stored), recorded."""
    from exllama_b200 import capi
    K, N, gs = SPREAD_SHAPE
    qw, qz, sc, x = spread_inputs(oracle)
    ref64 = oracle.q4_matmul_f64(x, qw, qz, sc)
    rms = float(np.sqrt(np.mean(ref64 ** 2)))
    tx = to_cuda(x)
    runs_ref = [r.astype(np.float64) for r in ref_golden()["spread_runs"]]
    q4 = capi.Q4(*to_cuda(qw.copy(), qz, sc))
    runs_mine = [capi.q4_matmul(tx, q4).cpu().numpy().astype(np.float64) for _ in range(3)]
    spread_ref = max(np.abs(runs_ref[i] - runs_ref[j]).max() for i in range(3) for j in range(i))
    spread_mine = max(np.abs(runs_mine[i] - runs_mine[j]).max() for i in range(3) for j in range(i))
    rec = {"shape": [1, K, N, gs], "rms_ref64": rms,
           "reference_max_run_to_run_diff": float(spread_ref), "reference_rms_err_vs_ref64": [float(np.sqrt(np.mean((r - ref64) ** 2))) for r in runs_ref],
           "ours_max_run_to_run_diff": float(spread_mine), "ours_rms_err_vs_ref64": [float(np.sqrt(np.mean((r - ref64) ** 2))) for r in runs_mine]}
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(rec, open(os.path.join(ROOT, "gpurun_out", "ref_spread.json"), "w"), indent=1)
    assert spread_mine == 0.0
    assert max(rec["ours_rms_err_vs_ref64"]) <= min(rec["reference_rms_err_vs_ref64"]) * 1.05 + 1e-9
