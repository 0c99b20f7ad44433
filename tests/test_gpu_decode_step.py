"""The whole-token persistent kernel (csrc/decode_step.cu) against (a) the oracle composition of the reference's decode
path -- rms_norm, q4_matmul, rope, cache update, attention, residual adds, silu*mul, final norm, lm_head, each restated
from the reference file:line the oracle cites -- and (b) this repo's own per-op kernels driven as model.py drives them
(DecodeStack.decode_step), on the same seeded synthetic GPTQ stack."""
import numpy as np
import pytest

from helpers import assert_close_ref64, mk_stack as _mk_stack, oracle_step as _oracle_step

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("gs,act", [(128, False), (32, False), (256, False), (128, True), (32, True)])
@pytest.mark.parametrize("past", [0, 1, 16, 37, 200])
def test_fused_step_vs_oracle_and_per_op_path(oracle, gs, act, past):
    import torch
    st = _mk_stack(1024, 2816, 2, 8, gs, 256, act=act)
    st.make_plan()
    info = st.dplan.info()
    assert info["grid"] >= 100 and info["ring_stages"] >= 8, info
    rng = np.random.default_rng(past + gs)
    x = (rng.standard_normal(st.shape.hidden) * 0.5).astype(np.float16)
    # (a) oracle, on a snapshot of the caches taken before anyone writes row `past`
    want_x, want_logits, rows = _oracle_step(oracle, st, x, past)
    snap = [(kc.clone(), vc.clone()) for kc, vc in zip(st.key_cache, st.value_cache)]
    # (b) per-op path (writes row `past` of the caches)
    hid = torch.from_numpy(x).cuda().view(1, 1, -1)
    ref_logits = st.decode_step(hid.clone(), past).cpu().numpy()
    per_op_rows = [(kc[0, :, past].cpu().numpy().copy(), vc[0, :, past].cpu().numpy().copy()) for kc, vc in zip(st.key_cache, st.value_cache)]
    for (kc, vc), (k0, v0) in zip(zip(st.key_cache, st.value_cache), snap):
        kc.copy_(k0); vc.copy_(v0)
    # fused
    logits = st.decode_step_fused(hid, past).cpu().numpy()
    torch.cuda.synchronize()
    got_x = st._plan_xout.cpu().numpy()
    # three matmuls deep per layer with fp16 rounding points in between: a few 1e-3 of the rms per layer
    assert_close_ref64(got_x, want_x.reshape(-1).astype(np.float64), rel=1e-2, rms=1e-2, what="final hidden vs oracle")
    assert_close_ref64(logits.reshape(-1), want_logits.reshape(-1), rel=1.5e-2, rms=1.5e-2, what="logits vs oracle")
    assert_close_ref64(logits.reshape(-1), ref_logits.reshape(-1).astype(np.float64), rel=1.5e-2, rms=1.5e-2, what="logits vs per-op path")
    for i, (kc, vc) in enumerate(zip(st.key_cache, st.value_cache)):
        k_new = kc[0, :, past].cpu().numpy(); v_new = vc[0, :, past].cpu().numpy()
        assert_close_ref64(k_new, rows[i][0].astype(np.float64), rel=1e-2, rms=1e-2, what=f"layer {i} new k row vs oracle")
        assert_close_ref64(v_new, rows[i][1].astype(np.float64), rel=1e-2, rms=1e-2, what=f"layer {i} new v row vs oracle")
        assert_close_ref64(k_new, per_op_rows[i][0].astype(np.float64), rel=1e-2, rms=1e-2, what=f"layer {i} new k row vs per-op")
        # nothing but row `past` was written
        mask = np.ones(st.max_seq, bool); mask[past] = False
        assert torch.equal(kc[0][:, mask], snap[i][0][0][:, mask]) and torch.equal(vc[0][:, mask], snap[i][1][0][:, mask])
    st.dplan.close(); st.close()


def test_fused_step_sequence_and_graph(oracle):
    """Five consecutive tokens (barrier generation, accumulator clean-up and the cache rows carry over between launches),
    then the same launch replayed from a CUDA graph: bit-identical KV rows are not required (fp32 atomics), logits agree."""
    import torch
    st = _mk_stack(1024, 2816, 3, 8, 128, 128, seed=5)
    st.make_plan()
    g = torch.Generator(device="cuda"); g.manual_seed(9)
    xs = [(torch.randn((1, 1, 1024), device="cuda", generator=g) * 0.5).half() for _ in range(5)]
    snap = [(kc.clone(), vc.clone()) for kc, vc in zip(st.key_cache, st.value_cache)]
    ref = [st.decode_step(x.clone(), 40 + i).clone() for i, x in enumerate(xs)]
    for (kc, vc), (k0, v0) in zip(zip(st.key_cache, st.value_cache), snap):
        kc.copy_(k0); vc.copy_(v0)
    got = [st.decode_step_fused(x, 40 + i).clone() for i, x in enumerate(xs)]
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(got, ref)):
        assert_close_ref64(a.cpu().numpy().reshape(-1), b.cpu().numpy().reshape(-1).astype(np.float64), rel=2e-2, rms=2e-2, what=f"token {i}")
    # graph replay of the last token
    x = xs[-1]
    side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        st.decode_step_fused(x, 44)
    torch.cuda.current_stream().wait_stream(side); torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        st.decode_step_fused(x, 44)
    for _ in range(3):
        gr.replay()
    torch.cuda.synchronize()
    assert_close_ref64(st._plan_logits.cpu().numpy().reshape(-1), got[-1].cpu().numpy().reshape(-1).astype(np.float64), rel=2e-3, rms=2e-3, what="graph replay")
    st.dplan.close(); st.close()


def test_fused_step_short_context_after_long_one(oracle):
    """ONE plan: a long context first (every slot of the attention-partial table gets written), then short contexts where some CTAs
    inside a head's CTA range own no attention unit (tests/test_decode_schedule.py: the hazard the CPU schedule proof found).
    Partials of the long context must not leak into the short contexts' softmax combine: exl_decode_step resets the table first."""
    import torch
    from exllama_b200 import capi
    st = _mk_stack(1024, 2816, 2, 8, 128, 256, seed=7)
    st.make_plan()
    g = torch.Generator(device="cuda"); g.manual_seed(21)
    snap = [(kc.clone(), vc.clone()) for kc, vc in zip(st.key_cache, st.value_cache)]

    def restore():
        for (kc, vc), (k0, v0) in zip(zip(st.key_cache, st.value_cache), snap):
            kc.copy_(k0); vc.copy_(v0)
    # 8 heads -> 56 CTAs take part in the attention phase; 16-position chunks: contexts 17 .. 96 leave some of them idle
    for past, extra in [(200, 0), (37, 1), (17, 1), (100, 0), (49, 1), (3, 0), (96, 1), (200, 0)]:
        x = (torch.randn((1, 1, 1024), device="cuda", generator=g) * 0.5).half()
        ref = st.decode_step(x.clone(), past).clone()
        restore()
        n0 = capi.launch_count()
        got = st.decode_step_fused(x, past).clone()
        torch.cuda.synchronize()
        assert capi.launch_count() - n0 == 1 + extra, (past, capi.launch_count() - n0)      # the table reset runs only where it is needed
        restore()
        assert_close_ref64(got.cpu().numpy().reshape(-1), ref.cpu().numpy().reshape(-1).astype(np.float64), rel=1.5e-2, rms=1.5e-2, what=f"logits at ctx {past}")
    st.dplan.close(); st.close()


def test_fused_step_7b_shape_long_context(oracle):
    """BASELINE shape (hidden 4096, inter 11008, 32 heads, vocab 32000) at ctx 1920, 2 layers: against the per-op path."""
    import torch
    st = _mk_stack(4096, 11008, 2, 32, 128, 2048, vocab=32000, seed=11)
    st.make_plan()
    x = (torch.randn((1, 1, 4096), device="cuda") * 0.5).half()
    snap = [(kc.clone(), vc.clone()) for kc, vc in zip(st.key_cache, st.value_cache)]
    ref = st.decode_step(x.clone(), 1920).clone()
    for (kc, vc), (k0, v0) in zip(zip(st.key_cache, st.value_cache), snap):
        kc.copy_(k0); vc.copy_(v0)
    got = st.decode_step_fused(x, 1920)
    torch.cuda.synchronize()
    assert torch.isfinite(got).all()
    assert_close_ref64(got.cpu().numpy().reshape(-1), ref.cpu().numpy().reshape(-1).astype(np.float64), rel=1.5e-2, rms=1.5e-2, what="7B-shape logits")
    st.dplan.close(); st.close()


def test_fused_step_act_order_13b_shape(oracle):
    """BASELINE config 3 shape (hidden 5120, inter 13824, 40 heads, act-order), 2 layers at ctx 1920: against the per-op path."""
    import torch
    st = _mk_stack(5120, 13824, 2, 40, 128, 2048, vocab=32000, seed=13, act=True)
    st.make_plan()
    x = (torch.randn((1, 1, 5120), device="cuda") * 0.5).half()
    snap = [(kc.clone(), vc.clone()) for kc, vc in zip(st.key_cache, st.value_cache)]
    ref = st.decode_step(x.clone(), 1920).clone()
    for (kc, vc), (k0, v0) in zip(zip(st.key_cache, st.value_cache), snap):
        kc.copy_(k0); vc.copy_(v0)
    got = st.decode_step_fused(x, 1920)
    torch.cuda.synchronize()
    assert torch.isfinite(got).all()
    assert_close_ref64(got.cpu().numpy().reshape(-1), ref.cpu().numpy().reshape(-1).astype(np.float64), rel=1.5e-2, rms=1.5e-2, what="13B-shape act-order logits")
    st.dplan.close(); st.close()
