"""CPU proof of the persistent decode kernel's static schedule (exllama_b200/csrc/decode_step_sched.h).

The header is the one decode_step.cu includes; tests/decode_sched_check.cpp compiles it with g++ and checks, for every
BASELINE shape (SURVEY.md 8), tensor-parallel shard, grid size and context length: the unit partition of every phase, the
inverse map used by the attention combine, the attention partial-slot table, the act-order staging slots, the lm_head
coverage and the shared-memory plan.  On the GPU a schedule mistake is a trapped launch or a stale partial; here it is a
failed assertion with the offending (context length, CTA, head).
"""
import ctypes
import os
import subprocess

import pytest

from exllama_b200.shapes import SHAPES
from exllama_b200.tp import plan_shards

HERE = os.path.dirname(os.path.abspath(__file__))
SMEM_OPTIN = 232448          # cudaDevAttrMaxSharedMemoryPerBlockOptin on sm_100 (227 KB)
SMS = 148


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("sched") / "libdecode_sched_check.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wall", "-Werror",
                           os.path.join(HERE, "decode_sched_check.cpp"), "-o", so])
    lib = ctypes.CDLL(so)
    lib.ds_check.restype = ctypes.c_int
    lib.ds_check.argtypes = [ctypes.c_int] * 9 + [ctypes.c_longlong, ctypes.c_char_p, ctypes.c_int, ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_int)]
    lib.ds_plan.restype = ctypes.c_int
    lib.ds_plan.argtypes = [ctypes.c_int] * 6 + [ctypes.c_longlong, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_int)]
    return lib


def check(lib, H, HQ, I, heads, vocab, grid, past_lo, past_hi, act, counts=None):
    msg = ctypes.create_string_buffer(512)
    gaps, resets = ctypes.c_longlong(), ctypes.c_int()
    rc = lib.ds_check(H, HQ, I, heads, vocab, grid, past_lo, past_hi, int(act), SMEM_OPTIN, msg, len(msg), ctypes.byref(gaps), ctypes.byref(resets))
    if counts is not None:
        counts["gaps"], counts["resets"] = gaps.value, resets.value
    return rc, msg.value.decode()


def local_shapes(name, tp, groupsize=128):
    """(hidden, local attention width, local intermediate width, local heads) of every rank."""
    s = SHAPES[name]
    plan = plan_shards(s.hidden, s.inter, s.heads, s.head_dim, groupsize, tp)
    out = []
    for r in range(tp):
        c0, c1 = plan.head_cols[r]
        i0, i1 = plan.inter_cols[r]
        out.append((s.hidden, c1 - c0, i1 - i0, plan.heads[r]))
    return sorted(set(out))


# BASELINE configs: 7B (seq 2048), 13B act-order, 33B g32 act-order TP2/4, 65B TP8 seq 4096 -- plus every other split that divides
CASES = [(n, tp) for n in ("7b", "13b", "33b", "65b") for tp in (1, 2, 4, 8) if SHAPES[n].heads % tp == 0]


@pytest.mark.parametrize("name,tp", CASES)
def test_schedule_every_context_length(lib, name, tp):
    gs = 32 if name == "33b" else 128
    max_seq = 4096 if name == "65b" else 2048
    for (H, HQ, I, heads) in local_shapes(name, tp, gs):
        rc, msg = check(lib, H, HQ, I, heads, SHAPES[name].vocab, SMS, 0, max_seq - 1, act=False)
        assert rc == 0, f"{name} tp{tp} local {(H, HQ, I, heads)}: {msg}"


@pytest.mark.parametrize("name", ["7b", "13b", "33b", "65b"])
def test_schedule_act_order_single_gpu(lib, name):
    # act-order runs in the step kernel on one GPU only: two staging slots, a wider shared-memory plan
    s = SHAPES[name]
    rc, msg = check(lib, s.hidden, s.hidden, s.inter, s.heads, s.vocab, SMS, 0, 2047, act=True)
    assert rc == 0, f"{name} act-order: {msg}"


@pytest.mark.parametrize("grid", [52, 64, 100, 132, 147])
def test_schedule_other_grids(lib, grid):
    # EXL_DS_GRID (bring-up) and parts with fewer SMs: the schedule must hold for any grid >= heads
    for name in ("7b", "33b"):
        s = SHAPES[name]
        if s.heads > grid:
            continue
        rc, msg = check(lib, s.hidden, s.hidden, s.inter, s.heads, s.vocab, grid, 0, 600, act=False)
        assert rc == 0, f"{name} grid {grid}: {msg}"


def test_schedule_no_head_and_tiny(lib):
    # the tiny shapes of tests/test_gpu_decode_step.py, tests/test_gpu_decode_step_variants.py and __graft_entry__.smoke();
    # a plan without lm_head; hidden = inter (one quantisation group per matrix); odd lm_head chunks per row (H 1536) with a
    # vocabulary that leaves a partial last head stage (2052 * 3 % 8 != 0)
    for (H, I, heads, vocab) in [(1024, 2816, 8, 0), (1024, 2816, 8, 512), (512, 1536, 4, 256), (2048, 5632, 16, 32000),
                                 (1024, 2816, 8, 2048), (1024, 1024, 8, 2048), (2048, 2048, 16, 2048), (1536, 4096, 12, 2052),
                                 (1536, 4096, 12, 2048)]:
        rc, msg = check(lib, H, heads * 128, I, heads, vocab, SMS, 0, 300, act=False)
        assert rc == 0, f"{(H, I, heads, vocab)}: {msg}"
        rc, msg = check(lib, H, heads * 128, I, heads, vocab, SMS, 0, 300, act=True)
        assert rc == 0, f"act {(H, I, heads, vocab)}: {msg}"
    # the small shape on the grids the GPU tests set through EXL_DS_GRID, every context of its 256-position cache
    for grid in (100, 132):
        for act in (False, True):
            rc, msg = check(lib, 1024, 1024, 2816, 8, 2048, grid, 0, 255, act=act)
            assert rc == 0, f"grid {grid} act {act}: {msg}"


def test_checker_rejects_bad_shapes(lib):
    rc, msg = check(lib, 4096 + 128, 4096, 11008, 32, 32000, SMS, 0, 4, act=False)      # hidden % 512
    assert rc == 1 and "multiples" in msg
    rc, msg = check(lib, 4096, 4096, 11008, 32, 32000, 16, 0, 4, act=False)            # more heads than CTAs
    assert rc == 1 and "heads" in msg
    rc, msg = check(lib, 32768, 32768, 4 * 32768, 256, 32000, 256, 0, 4, act=False)    # too wide for the shared-memory plan
    assert rc == 1 and "P7" in msg


def test_plan_sizes(lib):
    """Ring depth and shared-memory bytes of the BASELINE shapes (DESIGN.md 3c: 7B 16 stages / 222 KB; the wider models 12)."""
    depth, smem, slots = ctypes.c_int(), ctypes.c_longlong(), ctypes.c_int()
    want = {"7b": 4, "13b": 3, "33b": 3, "65b": 3}
    for name, d in want.items():
        s = SHAPES[name]
        lib.ds_plan(s.hidden, s.hidden, s.inter, s.heads, SMS, 0, SMEM_OPTIN, ctypes.byref(depth), ctypes.byref(smem), ctypes.byref(slots))
        assert depth.value >= 2 and smem.value + 2048 <= SMEM_OPTIN
        assert depth.value == d, (name, depth.value)
        assert slots.value == (SMS // s.heads + 2 if SMS < 7 * s.heads else 9)


def test_attention_table_reset_is_confined_to_short_contexts(lib):
    """Idle CTAs inside a head's CTA range (stale partial slots) exist only at short contexts, exactly where exl_decode_step resets
    the table; the steady state (every CTA has attention work) launches nothing extra."""
    s = SHAPES["7b"]
    c = {}
    rc, msg = check(lib, s.hidden, s.hidden, s.inter, s.heads, s.vocab, SMS, 0, 2047, False, c)
    assert rc == 0, msg
    assert c["gaps"] > 0                      # the hazard is real (found by this test before the reset existed) ...
    assert c["resets"] == 48                  # ... and confined: 32 heads x nph units < 148 CTAs, nph >= 2 -> contexts 17 .. 64
    rc, msg = check(lib, s.hidden, s.hidden, s.inter, s.heads, s.vocab, SMS, 65, 2047, False, c)
    assert rc == 0 and c["gaps"] == 0 and c["resets"] == 0
