"""TEST INFRASTRUCTURE — loader for the committed golden fixtures (tests/golden/*.pt)."""
import math
import os

import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def load_golden(name):
    return torch.load(os.path.join(GOLDEN_DIR, name), map_location="cpu", weights_only=False)


def sample_index(numel, n):
    """`n` distinct flat indices spread evenly over [0, numel): i * a mod numel for i < n, with `a` the integer nearest
    numel / golden ratio that is coprime to numel.  Integer arithmetic only, so the sample is the same on every machine
    and library version.  Full-size outputs are stored as their values at these indices to keep each fixture small."""
    if n >= numel:
        return torch.arange(numel)
    a = max(1, round(numel * 0.6180339887498949))
    while math.gcd(a, numel) != 1:
        a += 1
    return torch.arange(n, dtype=torch.int64) * a % numel


def sample_flat(x, n):
    """The values of `x` (any shape, any device) at sample_index(x.numel(), n), as a 1-D CPU tensor."""
    return x.detach().flatten().cpu()[sample_index(x.numel(), n)]
