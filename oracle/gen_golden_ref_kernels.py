"""Generates tests/golden/ref_kernels.npz: outputs of the REFERENCE's own CUDA kernels (oracle/_ref/libexllama_ref.so,
compiled from its sources for sm_100a by oracle/Makefile) on the seeded inputs of tests/test_gpu_ref_pin.py and
tests/test_gpu_q4_matmul.py, which build those inputs with the functions imported below.  Outputs of more than 2048
elements are stored at the helpers.sample_idx positions.  The properties of the reference that the tests do not need
stored (its cache layout, x left untouched by q4_attn) are asserted here.

Needs a B200 and oracle/_ref/ (make -C oracle ref):  python oracle/gen_golden_ref_kernels.py [OUT.npz]"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from helpers import REF_GOLDEN, RefLib, sample_idx, to_cuda  # noqa: E402
from oracle import oracle as O  # noqa: E402
import test_gpu_q4_matmul as Q  # noqa: E402
import test_gpu_ref_pin as P  # noqa: E402


def flat(t):
    a = t.cpu().numpy().reshape(-1) if torch.is_tensor(t) else np.asarray(t).reshape(-1)
    return a[sample_idx(a.size)]


def q4(ref, t):
    qw, qz, sc, g = t
    return ref.make_q4(*to_cuda(qw.copy(), qz, sc), g)


def main(path):
    torch.cuda.set_device(0)
    ref = RefLib()
    ref.prepare_buffers(inter=11008, max_rows=256, dq_numel=4096 * 11008)
    out = {}
    for rows, dim in P.RMS_CASES:
        tx, tw = to_cuda(*P.rms_norm_inputs(rows, dim))
        t = torch.empty_like(tx)
        torch.cuda.synchronize()
        ref.lib.ref_rms_norm(tx.data_ptr(), tw.data_ptr(), t.data_ptr(), 1e-6, rows, dim, 0); ref.sync()
        out[f"rms_norm_{rows}_{dim}"] = flat(t)
    for bsz, q_len, heads, hd, past in P.ROPE_CASES:
        x, sin, cos = P.rope_inputs(bsz, q_len, heads, hd, past)
        tx, ts, tc = to_cuda(x.copy(), sin, cos)
        torch.cuda.synchronize()
        ref.lib.ref_rope(tx.data_ptr(), ts.data_ptr(), tc.data_ptr(), bsz, q_len * heads, hd, heads, past); ref.sync()
        out[f"rope_{bsz}_{q_len}_{heads}_{hd}_{past}"] = flat(tx)
    for i, (x, perm) in enumerate(P.column_remap_inputs()):
        tx, tm = to_cuda(x, perm.view(np.int32))
        t = torch.empty_like(tx)
        torch.cuda.synchronize()
        ref.lib.ref_column_remap(tx.data_ptr(), t.data_ptr(), x.shape[0], x.shape[1], tm.data_ptr()); ref.sync()
        out[f"column_remap_{i}"] = flat(t)
    for i, (x, w) in enumerate(P.half_matmul_inputs()):
        tx, tw = to_cuda(x, w)
        t = torch.zeros((x.shape[0], w.shape[1]), dtype=torch.float16, device="cuda")
        torch.cuda.synchronize()
        ref.lib.ref_half_matmul_cublas(tx.data_ptr(), tw.data_ptr(), t.data_ptr(), x.shape[0], x.shape[1], w.shape[1], 0); ref.sync()
        out[f"half_matmul_cublas_{i}"] = flat(t)

    s = P.ATTN_SHAPE
    hidden, heads, hd, max_seq = s["hidden"], s["heads"], s["hd"], s["max_seq"]
    for act in (False, True):
        for q_len, past in P.ATTN_CASES:
            t, x, w, sin, cos = P.q4_attn_inputs(O, act, q_len)
            Qh, Kh, Vh = (q4(ref, t[n]) for n in ("q", "k", "v"))
            tx, tw, ts, tc = to_cuda(x.copy(), w, sin, cos)
            q = torch.zeros((1, q_len, hidden), dtype=torch.float16, device="cuda"); k = torch.zeros_like(q); v = torch.zeros_like(q)
            kc = torch.zeros((1, heads, max_seq, hd), dtype=torch.float16, device="cuda"); vc = torch.zeros_like(kc)
            torch.cuda.synchronize()
            ref.lib.ref_q4_attn(tx.data_ptr(), tw.data_ptr(), 1e-6, q.data_ptr(), k.data_ptr(), v.data_ptr(), Qh, Kh, Vh,
                                ts.data_ptr(), tc.data_ptr(), 1, q_len, hidden, hd, heads, heads, past,
                                kc.data_ptr(), vc.data_ptr(), max_seq, 0)
            ref.sync()
            q, k, v, kc, vc, xo = (a.cpu().numpy() for a in (q, k, v, kc, vc, tx))
            np.testing.assert_array_equal(xo, x)
            for tt in range(q_len):
                np.testing.assert_array_equal(kc[0, :, past + tt], k.reshape(q_len, heads, hd)[tt])
                np.testing.assert_array_equal(vc[0, :, past + tt], v.reshape(q_len, heads, hd)[tt])
            mask = np.ones(max_seq, bool); mask[past:past + q_len] = False
            assert not kc[0][:, mask].any() and not vc[0][:, mask].any()
            key = f"q4_attn_{int(act)}_{q_len}_{past}"
            out[key + "_q"], out[key + "_k"], out[key + "_v"] = q, k, v
        for rows in P.BLOCK_ROWS:
            t, x, attn, w = P.block_inputs(O, act, rows)
            Oh, Gh, Uh, Dh = (q4(ref, t[n]) for n in ("o", "gate", "up", "down"))
            ta, tw = to_cuda(attn, w)
            xr = to_cuda(x.copy()); torch.cuda.synchronize()
            ref.lib.ref_q4_attn_2(xr.data_ptr(), ta.data_ptr(), Oh, rows); ref.sync()
            out[f"block_{int(act)}_{rows}_attn_2"] = xr.cpu().numpy()
            xr = to_cuda(x.copy()); torch.cuda.synchronize()
            ref.lib.ref_q4_mlp(xr.data_ptr(), tw.data_ptr(), 1e-6, Gh, Uh, Dh, rows, hidden, 0); ref.sync()
            out[f"block_{int(act)}_{rows}_mlp"] = xr.cpu().numpy()

    qw, qz, sc, x = P.spread_inputs(O)
    h = q4(ref, (qw, qz, sc, None))
    tx = to_cuda(x)
    out["spread_runs"] = np.stack([ref.q4_matmul(tx, h, qw.shape[1], mode=0).cpu().numpy() for _ in range(3)])

    for M, K, N, gs, act in Q.REF_DECODE_CASES:
        qw, qz, sc, g_idx, x = Q.ref_decode_inputs(O, M, K, N, gs, act)
        tq, tz, ts = to_cuda(qw.copy(), qz, sc)
        h = ref.make_q4(tq, tz, ts, g_idx)
        key = f"q4_decode_{M}_{K}_{N}_{gs}_{int(act)}"
        out[key] = flat(ref.q4_matmul(to_cuda(x), h, N, mode=0))
        if act:
            out[key + "_qweight"] = flat(tq)          # make_q4 rewrote it into sequential order in place
    qw, qz, sc, x = Q.ref_recons_inputs(O)
    h = q4(ref, (qw, qz, sc, None))
    out["q4_recons"] = flat(ref.q4_matmul(to_cuda(x), h, qw.shape[1], mode=1))

    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes,", len(out), "arrays")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else REF_GOLDEN)
