"""Instantiations and edges of the persistent decode step (csrc/decode_step.cu) that tests/test_gpu_decode_step.py does not
reach: the groupsize-64 GEMV (gemv_t<2>), one quantisation group per matrix (gshift 30), odd lm_head chunks per row and a
partial last head stage, a plan without lm_head, the BASELINE widths against the float64 oracle, short contexts after a long
one at a wide shape, and grids other than one CTA per SM.

Each oracle case runs the fused step, the oracle composition (helpers.oracle_step) and the per-op path on the same snapshot of
the caches, with the tolerances of test_fused_step_vs_oracle_and_per_op_path.  It also checks a sharper condition on the final
hidden state and the new K / V rows: the fused step's rms error against the oracle is at most 1.25 x the per-op path's plus
1e-4 x rms.  Both paths round to fp16 at the same points, so a defect of the fused step alone shows up there long before it
reaches the 1e-2 tolerance."""
import numpy as np
import pytest

from helpers import assert_close_ref64, mk_stack, oracle_step
from helpers import sharper as _sharper

pytestmark = pytest.mark.gpu

SMALL = (1024, 2816, 8)          # hidden, inter, heads of the small test shape


def _restore(st, snap):
    for (kc, vc), (k0, v0) in zip(zip(st.key_cache, st.value_cache), snap):
        kc.copy_(k0); vc.copy_(v0)


def _run_vs_oracle(oracle, st, past, seed, what):
    """One token through the oracle, the per-op path and the fused step (plan already made) on the same cache snapshot."""
    import torch
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal(st.shape.hidden) * 0.5).astype(np.float16)
    want_x, want_logits, rows = oracle_step(oracle, st, x, past)
    snap = [(kc.clone(), vc.clone()) for kc, vc in zip(st.key_cache, st.value_cache)]
    # per-op path: updates its hidden state in place and writes row `past` of the caches
    hid = torch.from_numpy(x).cuda().view(1, 1, -1)
    ref_x = hid.clone()
    ref_out = st.decode_step(ref_x, past)
    ref_x = ref_x.cpu().numpy().reshape(-1)
    per_op_rows = [(kc[0, :, past].cpu().numpy().copy(), vc[0, :, past].cpu().numpy().copy()) for kc, vc in zip(st.key_cache, st.value_cache)]
    _restore(st, snap)
    out = st.decode_step_fused(hid, past)
    torch.cuda.synchronize()
    got_x = st._plan_xout.cpu().numpy()
    want_x = want_x.reshape(-1).astype(np.float64)
    assert_close_ref64(got_x, want_x, rel=1e-2, rms=1e-2, what=f"{what}: final hidden vs oracle")
    _sharper(got_x, ref_x, want_x, f"{what}: final hidden")
    if want_logits is not None:
        logits = out.cpu().numpy().reshape(-1)
        assert_close_ref64(logits, want_logits.reshape(-1), rel=1.5e-2, rms=1.5e-2, what=f"{what}: logits vs oracle")
        assert_close_ref64(logits, ref_out.cpu().numpy().reshape(-1).astype(np.float64), rel=1.5e-2, rms=1.5e-2, what=f"{what}: logits vs per-op path")
    mask = np.ones(st.max_seq, bool); mask[past] = False
    for i, (kc, vc) in enumerate(zip(st.key_cache, st.value_cache)):
        k_new = kc[0, :, past].cpu().numpy(); v_new = vc[0, :, past].cpu().numpy()
        k_want, v_want = rows[i][0].astype(np.float64), rows[i][1].astype(np.float64)
        assert_close_ref64(k_new, k_want, rel=1e-2, rms=1e-2, what=f"{what}: layer {i} new k row vs oracle")
        assert_close_ref64(v_new, v_want, rel=1e-2, rms=1e-2, what=f"{what}: layer {i} new v row vs oracle")
        assert_close_ref64(k_new, per_op_rows[i][0].astype(np.float64), rel=1e-2, rms=1e-2, what=f"{what}: layer {i} new k row vs per-op")
        _sharper(k_new, per_op_rows[i][0], k_want, f"{what}: layer {i} new k row")
        _sharper(v_new, per_op_rows[i][1], v_want, f"{what}: layer {i} new v row")
        # nothing but row `past` was written
        assert torch.equal(kc[0][:, mask], snap[i][0][0][:, mask]) and torch.equal(vc[0][:, mask], snap[i][1][0][:, mask])


@pytest.mark.parametrize("act", [False, True])
@pytest.mark.parametrize("past", [0, 15, 31, 200, 255])
def test_groupsize_64(oracle, act, past):
    """gemv_t<2> (two 32-k units per quantisation segment); past 255 writes the last row of a 256-position cache."""
    H, I, heads = SMALL
    st = mk_stack(H, I, 2, heads, 64, 256, act=act, seed=17)
    st.make_plan()
    _run_vs_oracle(oracle, st, past, seed=past + 64, what=f"g64 act{act} past {past}")
    st.dplan.close(); st.close()


@pytest.mark.parametrize("act", [False, True])
@pytest.mark.parametrize("hidden,heads", [(1024, 8), (2048, 16)])
def test_one_group_per_matrix(oracle, hidden, heads, act):
    """hidden = inter = groupsize: every matrix has one quantisation group (the plan's gshift 30)."""
    st = mk_stack(hidden, hidden, 2, heads, hidden, 256, act=act, seed=19)
    st.make_plan()
    _run_vs_oracle(oracle, st, 100, seed=hidden, what=f"one group H{hidden} act{act}")
    st.dplan.close(); st.close()


@pytest.mark.parametrize("vocab", [2052, 2048])
def test_head_odd_chunks_per_row(oracle, vocab):
    """H 1536: 3 lm_head chunks of 1 KB per row, so rows straddle the chunk pairs of a warp; vocab 2052 leaves a partial last
    stage of the 8-chunk head ring (2052 * 3 % 8 == 4)."""
    st = mk_stack(1536, 4096, 2, 12, 128, 256, vocab=vocab, seed=23)
    st.make_plan()
    _run_vs_oracle(oracle, st, 77, seed=vocab, what=f"H1536 vocab {vocab}")
    st.dplan.close(); st.close()


def test_plan_without_head(oracle):
    """make_plan(with_head=False): the step ends with the last layer's residual; _plan_xout against the oracle."""
    H, I, heads = SMALL
    st = mk_stack(H, I, 2, heads, 128, 256, seed=29, with_head=False)
    st.make_plan(with_head=False)
    assert st.dplan.vocab == 0 and st._plan_logits is None
    _run_vs_oracle(oracle, st, 150, seed=29, what="no head")
    st.dplan.close(); st.close()


BASELINE = [  # (name, hidden, inter, heads, groupsize, act_order, max_seq, past, ring stages per the CPU plan or None)
    ("7b", 4096, 11008, 32, 128, False, 2048, 2047, 16),
    ("13b", 5120, 13824, 40, 128, True, 2048, 1920, None),
    ("33b", 6656, 17920, 52, 32, True, 2048, 1000, None),
    ("65b", 8192, 22016, 64, 128, False, 4096, 4095, 12),
]


@pytest.mark.parametrize("name,hidden,inter,heads,gs,act,max_seq,past,stages", BASELINE)
def test_baseline_width_vs_oracle(oracle, name, hidden, inter, heads, gs, act, max_seq, past, stages):
    """Two layers at each BASELINE width against the float64 oracle (not only against this project's per-op path)."""
    st = mk_stack(hidden, inter, 2, heads, gs, max_seq, vocab=32000, act=act, seed=31)
    st.make_plan()
    info = st.dplan.info()
    if stages is not None:
        assert info["ring_stages"] == stages, info       # tests/test_decode_schedule.py::test_plan_sizes
    else:
        assert info["ring_stages"] >= 8, f"{name} act-order ring stages {info['ring_stages']} ({info})"
    _run_vs_oracle(oracle, st, past, seed=len(name) + past, what=f"{name} g{gs} act{act} past {past} ({info['ring_stages']} stages)")
    st.dplan.close(); st.close()


def test_short_contexts_after_long_65b_width(oracle):
    """One 65B-width plan: past 4000 (every slot of the attention-partial table written), then short contexts at and around the
    16-position chunk edges, then 4000 again, each against the per-op path.  64 heads leave a different set of idle attention
    CTAs at short contexts than the small shape's 8."""
    import torch
    st = mk_stack(8192, 22016, 2, 64, 128, 4096, vocab=32000, seed=37)
    st.make_plan()
    g = torch.Generator(device="cuda"); g.manual_seed(41)
    snap = [(kc.clone(), vc.clone()) for kc, vc in zip(st.key_cache, st.value_cache)]
    for past in [4000, 16, 32, 47, 63, 64, 4000]:
        x = (torch.randn((1, 1, 8192), device="cuda", generator=g) * 0.5).half()
        ref_x = x.clone()
        ref = st.decode_step(ref_x, past).clone()
        _restore(st, snap)
        got = st.decode_step_fused(x, past).clone()
        torch.cuda.synchronize()
        got_x = st._plan_xout.cpu().numpy()
        _restore(st, snap)
        assert_close_ref64(got_x, ref_x.cpu().numpy().reshape(-1).astype(np.float64), rel=1e-2, rms=1e-2, what=f"final hidden at past {past}")
        assert_close_ref64(got.cpu().numpy().reshape(-1), ref.cpu().numpy().reshape(-1).astype(np.float64), rel=1.5e-2, rms=1.5e-2, what=f"logits at past {past}")
    st.dplan.close(); st.close()


@pytest.mark.parametrize("grid", [100, 132])
@pytest.mark.parametrize("past", [16, 200])
def test_other_grids(oracle, monkeypatch, grid, past):
    """EXL_DS_GRID (read at plan creation): fewer CTAs than SMs, so every phase partitions its units differently."""
    H, I, heads = SMALL
    monkeypatch.setenv("EXL_DS_GRID", str(grid))
    st = mk_stack(H, I, 2, heads, 128, 256, seed=43)
    st.make_plan()
    assert st.dplan.info()["grid"] == grid
    _run_vs_oracle(oracle, st, past, seed=grid + past, what=f"grid {grid} past {past}")
    st.dplan.close(); st.close()
