"""Shared helpers for the parity tests (CPU side)."""
import gzip
import json
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def load_golden(name):
    z = np.load(os.path.join(GOLD, name))
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}
    rest = {k: z[k] for k in z.files if not k.startswith("sd.")}
    return sd, rest


def load_golden_json(name):
    with open(os.path.join(GOLD, name)) as f:
        return json.load(f)


def golden_bpe_vocab(directory):
    """Write a BPE merge table of CLIP's length to `directory` and return its path.  It holds the merges that the reference tokenizer applies to
    the golden captions (golden/bpe_merges.json) at their ranks in CLIP's table, and an inert pair at every other rank (U+2400 is outside the
    byte alphabet, so no text forms it).  Lowest-rank-first merging only ever applies pairs of the stored set, so these captions get CLIP's token
    ids, and the vocabulary keeps CLIP's size."""
    g = load_golden_json("bpe_merges.json")
    lines = [f"␀{r} ␀" for r in range(g["n_merges"])]
    for r, a, b in g["merges"]:
        lines[r] = f"{a} {b}"
    path = os.path.join(str(directory), "bpe_golden.txt.gz")
    with gzip.open(path, "wt", encoding="utf-8") as f:
        f.write("\n".join(["#version: 0.2"] + lines) + "\n")
    return path


def portable_uniform(seed, shape):
    rng = np.random.Generator(np.random.Philox(seed))
    return torch.from_numpy(rng.random(size=tuple(shape), dtype=np.float32))


def sampler_case_inputs(case, B=2, K=256, L=265):
    """Must stay identical to oracle/gen_golden.py:sampler_case_inputs (inputs are regenerated, not stored)."""
    scale = [1.0, 6.0, 40.0, 2.0, 12.0][case % 5]
    logits = (portable_uniform(100 + case, (B, K, L)) - 0.5) * scale
    u = portable_uniform(200 + case, (B, K + 1, L))
    t_pair = [(99, 99), (57, 12), (1, 1), (0, 0), (98, 33)][case % 5]
    t = torch.tensor([t_pair[i % 2] for i in range(B)], dtype=torch.long)
    ids = (portable_uniform(300 + case, (B, L)) * K).long().clamp(max=K - 1)
    masked = portable_uniform(400 + case, (B, L)) < ([1.1, 0.35, 0.05, 0.02, 0.9][case % 5])
    x_t = torch.where(masked, torch.full_like(ids, K), ids)
    return logits, x_t, t, u


def rel_err(a, b):
    """max |a-b| / max|b|  -- the 'relative' of north_star's 1e-3 (relative to the tensor's scale)."""
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))
