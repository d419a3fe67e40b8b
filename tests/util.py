"""Deterministic synthetic inputs shared by the golden generator, the tests and the bench."""
from __future__ import annotations

import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def make_inputs(seed: int, B: int, T: int, hp, ragged: bool = False, gen_only: bool = False):
    """SURVEY.md §8d input recipe: ppg, vec ~ N(0,1); integer-Hz f0 in [100,500] with an unvoiced
    span (the reference reads F0 from a CSV of ints, pitch/inference.py:113-119); spk ~ 0.05*N(0,1)
    (scale of the shipped singer embeddings); every random draw of the reference as a tensor."""
    g = torch.Generator().manual_seed(seed)
    hop = int(np.prod(list(hp.gen.upsample_rates)))
    L = T * hop
    d = {}
    d["pit"] = torch.randint(100, 501, (B, T), generator=g).float()
    u0 = max(1, int(0.30 * T))
    d["pit"][:, u0:u0 + max(1, int(0.15 * T))] = 0.0
    d["spk"] = torch.randn(B, hp.vits.spk_dim, generator=g) * 0.05
    d["rand_ini"] = torch.rand(B, 11, generator=g)
    d["noise"] = torch.randn(B, L, 11, generator=g)
    if gen_only:
        d["z"] = torch.randn(B, hp.gen.upsample_input, T, generator=g)
    else:
        d["ppg"] = torch.randn(B, T, hp.vits.ppg_dim, generator=g)
        d["vec"] = torch.randn(B, T, hp.vits.vec_dim, generator=g)
        d["eps"] = torch.randn(B, hp.vits.inter_channels, T, generator=g)
        if ragged:
            lens = torch.randint(int(0.6 * T), T + 1, (B,), generator=g)
            lens[0] = T
            d["ppg_l"] = lens.long()
        else:
            d["ppg_l"] = torch.full((B,), T, dtype=torch.long)
    return d


def seeded_sample(x, k: int = 8192):
    """A fixed, seeded sample of k values of x (flattened; all of x when it has at most k): the same positions
    for every x of one size, so that samples of two runs compare value for value.  Golden fixtures and
    `bench.py --dump-outputs` keep large outputs small this way.  The positions are random so that no stride
    of the output's layout (channels, up-sampling phases) is left out."""
    flat = torch.as_tensor(x).reshape(-1)
    if flat.numel() <= k:
        return flat
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:k].sort().values
    return flat[idx]


def launched_kernels(fn) -> set:
    """Names of the kernels the device launches during `fn()`, read from svcb_timing_report with kernel
    timing switched on for the call."""
    import torch
    from whisper_vits_svc_b200 import _lib
    lib = _lib.load()
    lib.svcb_timing_enable(1)
    try:
        fn()
        torch.cuda.synchronize()
        rep = lib.svcb_timing_report().decode()
    finally:
        lib.svcb_timing_enable(0)
    return {line.split()[0] for line in rep.splitlines() if line.strip()}


def max_abs(a, b):
    return float((torch.as_tensor(a).float().cpu() - torch.as_tensor(b).float().cpu()).abs().max())


def rel_l2(a, b):
    a = torch.as_tensor(a).float().cpu()
    b = torch.as_tensor(b).float().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))
