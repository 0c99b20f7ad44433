"""Generates tests/golden/rep_penalty_ref.npz and tests/golden/rep_penalty_ref_random.npz by running the REFERENCE's own
rep_penalty.cpp (compiled into oracle/_ref/librep_penalty_ref.so from the reference's sources; see oracle/Makefile).
The second file holds, for the random cases of tests/test_oracle.py, the mask entries that are not 1 and the logits
apply_rep_penalty changed.
Run where oracle/_ref/ is built:  python oracle/gen_golden_cpu.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from oracle import oracle as O  # noqa: E402
from test_oracle import rep_penalty_random_cases  # noqa: E402

assert O.ref_cpu_lib() is not None, "build oracle/_ref first (make -C oracle ref)"
rng = np.random.default_rng(20260922)
cases = [(16, 4, 1.15, 2, 2), (64, 40, 1.2, 8, 16), (1000, 300, 1.3, 64, 128), (50, 10, 1.25, -1, 0),
         (50, 7, 1.1, 0, 5), (4096, 512, 1.18, 256, 256), (100, 1, 1.5, 0, 0), (100, 30, 1.0, 10, 10)]
out = {"n_cases": len(cases)}
for i, (vocab, n, pmax, sustain, decay) in enumerate(cases):
    seq = rng.integers(0, vocab, size=n).astype(np.int64)
    if i == 0:
        seq = np.array([5, 7, 7, 9], dtype=np.int64)
    logits = rng.standard_normal(vocab).astype(np.float32)
    out[f"vocab_{i}"], out[f"pmax_{i}"], out[f"sustain_{i}"], out[f"decay_{i}"] = vocab, pmax, sustain, decay
    out[f"seq_{i}"], out[f"logits_{i}"] = seq, logits
    out[f"mask_{i}"] = O.rep_penalty(vocab, seq, pmax, sustain, decay, use_ref=True)
    out[f"applied_{i}"] = O.apply_rep_penalty(seq[None], pmax, sustain, decay, logits[None], use_ref=True)[0]
path = os.path.join(ROOT, "tests", "golden", "rep_penalty_ref.npz")
np.savez_compressed(path, **out)
print("wrote", path)

cols = {k: [] for k in ("params", "pmax", "mask_idx", "mask_val", "applied_idx", "applied_val")}
for vocab, seq, pmax, sustain, decay, lg in rep_penalty_random_cases():
    cols["params"].append([vocab, seq.size, sustain, decay]); cols["pmax"].append(pmax)
    mask = O.rep_penalty(vocab, seq, pmax, sustain, decay, use_ref=True)
    applied = O.apply_rep_penalty(seq[None], pmax, sustain, decay, lg, use_ref=True)[0]
    for name, got, base in (("mask", mask, 1.0), ("applied", applied, lg[0])):
        idx = np.flatnonzero(got != base)
        cols[name + "_idx"].append(idx); cols[name + "_val"].append(got[idx])
out = {"params": np.array(cols["params"]), "pmax": np.array(cols["pmax"])}
for name in ("mask", "applied"):        # per case: the entries that differ from 1 (mask) or from the input logits (applied)
    out[name + "_len"] = np.array([len(i) for i in cols[name + "_idx"]])
    out[name + "_idx"] = np.concatenate(cols[name + "_idx"]).astype(np.int16)      # vocab < 2000
    out[name + "_val"] = np.concatenate(cols[name + "_val"])
path = os.path.join(ROOT, "tests", "golden", "rep_penalty_ref_random.npz")
np.savez_compressed(path, **out)
print("wrote", path, os.path.getsize(path))
