"""Seeded parameter values and strided samples for fixtures that compare this package with the reference.

A fixture stores the reference's outputs, not its weights: the weights are drawn here from a seed, the same way by the
generator (oracle/gen_golden_live.py) and by the test, which keeps tests/golden/ small."""
import math

import torch


def seeded_state_dict(shapes, seed, gain=1.0):
    """{name: tensor} for {name: shape}, drawn in sorted-name order from one torch.Generator: matrices (and higher-rank
    weights) N(0, gain^2 / fan_in), positional tables N(0, 0.2^2), mixing coefficients (time_*) U(0, 1), 1-D weights
    1 + N(0, 0.1^2), 1-D biases N(0, 0.05^2)"""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for k in sorted(shapes):
        shape = tuple(int(s) for s in shapes[k])
        v = torch.randn(shape, generator=g)
        if "time_" in k:
            v = torch.rand(shape, generator=g)
        elif "pos_emb" in k:
            v = 0.2 * v
        elif len(shape) >= 2:
            v = v * (gain / math.sqrt(math.prod(shape[1:])))
        elif k.endswith("weight"):
            v = 1.0 + 0.1 * v
        else:
            v = 0.05 * v
        out[k] = v
    return out


def parse_shapes(entries):
    """{name: shape} from the "name=AxB" strings a fixture stores"""
    out = {}
    for e in entries:
        k, s = str(e).split("=")
        out[k] = tuple(int(x) for x in s.split("x")) if s else ()
    return out


def strided_sample(a, n=256):
    """every k-th element of the flattened array (numpy or torch), k chosen so that about n remain"""
    flat = a.reshape(-1)
    return flat[::max(1, flat.shape[0] // n)]
