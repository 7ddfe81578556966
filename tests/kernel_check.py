"""Helpers shared by the single-kernel GPU tests (test_gpu_encoder_kernels.py, test_gpu_decoder_kernels.py): the values a
kernel reads from an activation, the element-wise bound and the worst-error report.

FPNMT_KERNEL_ERRORS=<path> merges the worst error of each operator, as a fraction of its bound, into that JSON file (the
operators of the modules run earlier in the same or another session stay in it)."""
import json
import os

import numpy as np
import pytest
import torch

RTOL = {"bf16": 2.0 ** -8, "bf16x3": 2.0 ** -15}
WORST = {}


def record(op, value, bound):
    cur = WORST.get(op)
    if cur is None or value / bound > cur["worst"] / cur["bound"]:
        WORST[op] = {"worst": float(value), "bound": float(bound)}


def write_report():
    path = os.environ.get("FPNMT_KERNEL_ERRORS")
    if not path or not WORST:
        return
    merged = {}
    if os.path.exists(path):
        with open(path) as f:
            merged = json.load(f)
    merged.update(WORST)
    with open(path, "w") as f:
        json.dump(merged, f, indent=1, sort_keys=True)


@pytest.fixture(scope="module", autouse=True)
def error_report():
    """Import into a test module to write the report when the module's tests are done."""
    yield
    write_report()


def gen(seed):
    return torch.Generator().manual_seed(seed)


def q_act(x, prec):
    """The values a kernel reads from an activation stored from fp32 x: bf16(x), or hi + lo with hi = bf16(x) and
    lo = bf16(x - hi) (st_act), summed in fp32 as ld_act does."""
    x = x.float()
    hi = x.to(torch.bfloat16).float()
    if prec == "bf16":
        return hi
    return hi + (x - hi).to(torch.bfloat16).float()


def check_elementwise(op, y, ref, scale, rtol, atol, floor=0.0):
    """|y - ref| <= rtol |ref| + atol scale + floor everywhere, y finite."""
    y = y.double()
    assert bool(torch.isfinite(y).all()), "%s: %d non-finite outputs (never written?)" % (op, int((~torch.isfinite(y)).sum()))
    err = (y - ref).abs()
    bound = rtol * ref.abs() + atol * scale + floor
    ratio = err / bound.clamp_min(1e-300)
    worst = float(ratio.max())
    record(op, worst, 1.0)
    if worst > 1.0:
        i = int(ratio.flatten().argmax())
        idx = np.unravel_index(i, tuple(y.shape))
        raise AssertionError("%s: |y - ref| = %.3g > bound %.3g at %s (y %.8g, ref %.8g, scale %.3g); %d elements over" % (
            op, float(err.flatten()[i]), float(bound.flatten()[i]), idx, float(y.flatten()[i]), float(ref.flatten()[i]),
            float(torch.as_tensor(scale).expand_as(ref).flatten()[i]), int((ratio > 1).sum())))
