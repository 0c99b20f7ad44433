"""Every tile configuration of the tcgen05 prefill GEMM (csrc/q4_gemm_tc.cu) against float64.

exl_tc_gemm_launch chooses one of three CTA tiles from the problem size: 128x128 (<1,1,1>), 256x128 (<2,1,*>) and 256x256
(<2,2,*>), the last with its own dequant thread mapping (NT == 2).  The x-tile multicast variants (<2,*,2>, EXL_TC_MC=1) pad an
odd N-tile count with a CTA that works on out-of-range columns.  The first group of tests reaches each tile through the natural
selection rule at prefill shapes (the BASELINE prefill runs 256x256) and checks which one ran; the second forces each of the five
instantiations in a child process (the knobs are read once per process) on small ragged shapes.

B operand = the fp16-rounded reconstructed weights, accumulated in fp32 -> compared with the `recons` flavour of ref64 at the
helpers.assert_close_ref64 default tolerances (fp16 output rounding).  Large products are compared on a sample that holds the
first and last 8 rows / columns of every 128-wide sub-tile and all of a partial last tile (helpers.ref64_sampled: exact)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import ROOT, assert_close_ref64, ref64_sampled, tile_edge_sample, to_cuda

pytestmark = pytest.mark.gpu

SMS = 148      # the selection rule's tile-count thresholds are fractions of the SM count; the expected tiles below assume a B200

NATURAL = [  # (M, K, N, groupsize, act_order, expected tile)
    (1920, 4096, 4096, 128, False, "256x256"),      # BASELINE 7B prefill; the last 256-row tile is half empty
    (1920, 4096, 4224, 32, True, "256x256"),        # N % 256 == 128: the second N sub-tile of the last tile is wholly out of range
    (1921, 11008, 4104, 128, False, "256x256"),     # one row in the last M sub-tile; 8-column N tail; down_proj K
    (1920, 2048, 4096, 2048, False, "256x256"),     # one group per matrix (gs_shift32 = 30)
    (129, 4096, 11008, 128, False, "256x128"),      # the second M sub-tile holds one row
    (300, 2048, 9600, 64, True, "256x128"),         # groupsize 64, act-order
    (128, 4096, 11008, 128, False, "128x128"),      # M = 128 stays on the small tile
]


def _q4(capi, qw, qz, sc, g_idx):
    import torch
    tq, tz, ts = to_cuda(qw.copy(), qz, sc)
    return capi.Q4(tq, tz, ts, None if g_idx is None else torch.from_numpy(g_idx))


@pytest.mark.parametrize("M,K,N,gs,act,want", NATURAL)
def test_natural_tile_vs_ref64(oracle, M, K, N, gs, act, want):
    import torch
    from exllama_b200 import capi
    qw, qz, sc, g_idx = oracle.synth_q4(K, N, gs, act_order=act, seed=M + K + N)
    x = oracle.synth_x(M, K, seed=M)
    res = oracle.synth_x(M, N, seed=M + 1)
    q4 = _q4(capi, qw, qz, sc, g_idx)
    # q4_matmul sends a width that is not a multiple of 32 (the skinny kernel's unit) to the reconstruct + cuBLAS route at any M;
    # force_path=2 keeps such a width on the tcgen05 GEMM, whose launcher still chooses the tile by its own rule
    path = 0 if N % 32 == 0 else 2
    out = capi.q4_matmul(to_cuda(x), q4, force_path=path)
    torch.cuda.synchronize()
    assert capi.last_q4_path() == "tc_gemm"
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if sms == SMS:
        assert capi.last_tc_config() == want, (capi.last_tc_config(), want)
    out2 = to_cuda(res.copy())
    capi.q4_matmul(to_cuda(x), q4, out=out2, no_zero=True, force_path=path)
    torch.cuda.synchronize()
    assert capi.last_q4_path() == "tc_gemm"
    rows, cols = tile_edge_sample(M), tile_edge_sample(N)
    ref = ref64_sampled(x, qw, qz, sc, g_idx, rows, cols)
    what = f"tc_gemm M{M} K{K} N{N} g{gs} act{act} ({capi.last_tc_config()})"
    assert_close_ref64(out.cpu().numpy()[rows][:, cols], ref, what=what)
    # out += x.W: the float64 sum of the residual and the product (q4_matmul_f64 with acc_in adds the same two terms)
    ref2 = ref + res[rows][:, cols].astype(np.float64)
    assert_close_ref64(out2.cpu().numpy()[rows][:, cols], ref2, what=what + " accumulate")
    if sms != SMS:
        pytest.skip(f"tile choice not asserted: {sms} SMs (the expected tiles assume {SMS})")


# ---------------------------------------------------------------------------------------------------
# forced instantiations, one child process each
# ---------------------------------------------------------------------------------------------------

FORCED = [  # (EXL_TC_CFG, EXL_TC_MC, tile the launcher reports)
    ("1", "0", "128x128"),
    ("2", "0", "256x128"),
    ("2", "1", "256x128+mc"),
    ("3", "0", "256x256"),
    ("3", "1", "256x256+mc"),
]
# N-tile counts: 264 -> 3 (128-wide) / 2 (256-wide), 520 -> 5 / 3, 1160 -> 10 / 5: every multicast variant gets an odd count
SMALL_K = 1024     # 16 k-blocks: the 4-stage TMA ring and the B double buffer wrap several times
SMALL = [  # (M, N, groupsize, act_order)
    (129, 264, 128, False),
    (300, 520, 32, True),
    (129, 1160, 32, False),
    (300, 264, 128, True),
    (300, 1160, 128, False),
    (129, 520, 128, True),
]

CHILD = r"""
import sys
import numpy as np
import torch
from exllama_b200 import capi
d = dict(np.load(sys.argv[1]))
out = {}
for i in range(int(d["n"])):
    g = d.get(f"g{i}")
    qw = torch.from_numpy(d[f"qw{i}"]).cuda()
    q4 = capi.Q4(qw, torch.from_numpy(d[f"qz{i}"]).cuda(), torch.from_numpy(d[f"sc{i}"]).cuda(), None if g is None else torch.from_numpy(g))
    x = torch.from_numpy(d[f"x{i}"]).cuda()
    out[f"y{i}"] = capi.q4_matmul(x, q4, force_path=2).cpu().numpy()
    out[f"cfg{i}"] = np.array(capi.last_tc_config())
    acc = torch.from_numpy(d[f"r{i}"]).cuda()
    capi.q4_matmul(x, q4, out=acc, no_zero=True, force_path=2)
    out[f"ya{i}"] = acc.cpu().numpy()
    out[f"path{i}"] = np.array(capi.last_q4_path())
torch.cuda.synchronize()
np.savez(sys.argv[2], **out)
"""


@pytest.fixture(scope="module")
def small_cases(oracle, tmp_path_factory):
    """Inputs of the SMALL shapes (written once for every child) and their full float64 results."""
    path = str(tmp_path_factory.mktemp("tc_forced") / "inputs.npz")
    arrs, refs = {"n": np.array(len(SMALL))}, []
    for i, (M, N, gs, act) in enumerate(SMALL):
        qw, qz, sc, g_idx = oracle.synth_q4(SMALL_K, N, gs, act_order=act, seed=100 + i)
        x = oracle.synth_x(M, SMALL_K, seed=200 + i)
        res = oracle.synth_x(M, N, seed=300 + i)
        arrs.update({f"qw{i}": qw, f"qz{i}": qz, f"sc{i}": sc, f"x{i}": x, f"r{i}": res})
        if g_idx is not None:
            arrs[f"g{i}"] = g_idx
        refs.append((oracle.ref64_with_act_order(x, qw, qz, sc, g_idx, recons=True),
                     oracle.ref64_with_act_order(x, qw, qz, sc, g_idx, acc_in=res, recons=True)))
    np.savez(path, **arrs)
    return path, refs


@pytest.mark.parametrize("cfg,mc,want", FORCED)
def test_forced_tile_vs_ref64(small_cases, tmp_path, cfg, mc, want):
    inputs, refs = small_cases
    outputs = str(tmp_path / "outputs.npz")
    env = dict(os.environ, EXL_TC_CFG=cfg, EXL_TC_MC=mc)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", CHILD, inputs, outputs]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, f"child (EXL_TC_CFG={cfg} EXL_TC_MC={mc}) failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    got = dict(np.load(outputs))
    for i, (M, N, gs, act) in enumerate(SMALL):
        assert str(got[f"path{i}"]) == "tc_gemm"
        assert str(got[f"cfg{i}"]) == want, (str(got[f"cfg{i}"]), want)
        what = f"{want} M{M} K{SMALL_K} N{N} g{gs} act{act}"
        assert_close_ref64(got[f"y{i}"], refs[i][0], what=what)
        assert_close_ref64(got[f"ya{i}"], refs[i][1], what=what + " accumulate")
