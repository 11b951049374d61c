"""CPU checks of the forward-pass error model behind tests/test_gpu_forward.py (oracle/forward_bounds.py): the per-row bound
contains the rounding model of every path, and the normwise bar of precision 1 / 2 rejects an operand in the wrong format."""
import os
import sys

import numpy as np
import pytest

from oracle import ddpg_np as D
from oracle import forward_bounds as FB

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import precision_model as PM  # noqa: E402

STD = (4, 256, 48, 128)
HIGH = 2.5
FP32_BAR = 1e-5


def make_nets(seed, dims=STD):
    """The weight generator of tests/test_gpu_forward.py."""
    ns, l1, la, l2 = dims
    rng = np.random.default_rng(seed)
    ac, cr = D.init_actor(rng, ns, l1, l2), D.init_critic(rng, ns, l1, la, l2)
    D.randomize_bn(ac, rng, [("g1", "be1", "mu1", "var1"), ("g2", "be2", "mu2", "var2")])
    D.randomize_bn(cr, rng, [("gs", "bes", "mus", "vars"), ("ga", "bea", "mua", "vara"), ("g2", "be2", "mu2", "var2")])
    for p in (ac, cr):
        for k in p:
            if k.startswith("b") and not k.startswith("be"):
                p[k] = rng.normal(0, 0.05, p[k].shape).astype(np.float32)
    ac["W3"] *= 50
    cr["W3"] *= 300
    return ac, cr


def case(seed, R, critic, dims=STD):
    p = make_nets(seed, dims)[int(critic)]
    rng = np.random.default_rng(seed + 7)
    s = rng.normal(0, 2, (R, dims[0])).astype(np.float32).astype(np.float64)
    a = rng.uniform(-HIGH, HIGH, R).astype(np.float32).astype(np.float64)
    return p, s, a


def model(p, critic, s, a, sites):
    return FB.output(PM.Net(p, critic, sites).forward(s, a)[0], critic, HIGH)


def test_forward_path_follows_fused3_supported():
    assert FB.forward_path(STD, 1) == FB.forward_path(STD, 2) == "fused"
    assert FB.forward_path(STD, 0) == FB.forward_path(STD, 3) == "unfused"
    assert FB.forward_path((3, 256, 16, 128), 2) == "fused"
    for dims in ((4, 256, 56, 128), (4, 256, 64, 128), (5, 256, 48, 128), (4, 256, 48, 96), (4, 264, 48, 128), (4, 256, 40, 128)):
        assert FB.forward_path(dims, 2) == "unfused"
        assert FB.operand_formats(dims, 2) == ("bf16", "bf16")      # operand_format(2): no fp16 outside the fused kernels
    assert FB.operand_formats(STD, 2) == ("fp16", "fp16") and FB.operand_formats(STD, 1) == ("bf16", "bf16")


def test_fp16_forward_operands_have_a_subnormal_floor():
    """Unscaled fp16 rounds values below 2^-14 on a fixed grid of 2^-24: the error is absolute there, at most 2^-25."""
    x = np.geomspace(1e-12, 1e-3, 10_001)
    err = np.abs(PM.rnd(x, "fp16sat") - x.astype(np.float32))
    assert np.all(err <= FB.U_FMT["fp16"] * x + FB.FP16_FLOOR)
    assert np.max(err[x < 2.0 ** -14] / x[x < 2.0 ** -14]) > 10 * FB.U_FMT["fp16"]
    assert PM.rnd(np.array([1e6, -1e6]), "fp16sat").tolist() == [65504.0, -65504.0]


@pytest.mark.parametrize("dims,precision", [(STD, 1), (STD, 2), ((4, 256, 64, 128), 1), ((4, 256, 64, 128), 2), (STD, 0), (STD, 3)],
                         ids=["fused-bf16", "fused-fp16", "unfused-bf16-p1", "unfused-bf16-p2", "fp32", "split3"])
@pytest.mark.parametrize("critic", [False, True], ids=["actor", "critic"])
def test_bound_contains_the_rounding_model(dims, precision, critic):
    """tools/precision_model.Net with the operands of the path rounded as the kernels round them stays inside the bound on
    every row: 20 seeds at R = 64, 2 at R = 16384."""
    sites = FB.model_sites(dims, precision)
    for seed, R in [(sd, 64) for sd in range(20)] + [(100, 16384), (101, 16384)]:
        p, s, a = case(seed, R, critic, dims)
        bnd, ref = FB.row_bound(p, critic, s, a, dims=dims, precision=precision, high=HIGH)
        err = np.abs(model(p, critic, s, a, sites) - ref)
        assert np.all(np.isfinite(bnd)) and np.all(err <= bnd), (seed, R, float(np.max(err / bnd)))


WRONG = {"r1 in bf16": dict(r1="bf16"), "W2' in bf16": dict(W2f="bf16"), "layer 1 without lo": dict(l1="bf16")}


@pytest.mark.parametrize("wrong", list(WRONG), ids=["r1-bf16", "W2f-bf16", "layer1-no-lo"])
@pytest.mark.parametrize("critic", [False, True], ids=["actor", "critic"])
def test_precision2_bar_rejects_a_wrong_operand_format(wrong, critic):
    """The normwise bar of tests/test_gpu_forward.py at precision 2 is 2 E + 1e-5, E the model's error with the kernel's sites.
    A model that rounds one operand more coarsely than the kernel must fail it from 64 rows up (the error of a handful of rows is
    a draw of a few rounding sums, so at R = 1 the bar is a sanity check rather than a test of the format)."""
    sites = FB.model_sites(STD, 2)
    bad = dict(sites, **WRONG[wrong])
    for seed, R in [(sd, 64) for sd in range(10)] + [(20, 129), (100, 4133), (101, 16384)]:
        p, s, a = case(seed, R, critic)
        ref = FB.output(FB.exact(p, critic, s, a)[0], critic, HIGH)
        bar = 2 * FB.normwise(model(p, critic, s, a, sites), ref) + FP32_BAR
        e = FB.normwise(model(p, critic, s, a, bad), ref)
        assert e > bar, (seed, R, e, bar)


def test_bars_stay_within_twice_the_model():
    """The precision 1 / 2 bar is tied to the model's own error: at the fp32 floor alone it could not reject anything, and the
    floor is far below the fp16 model error it is added to."""
    for critic in (False, True):
        p, s, a = case(3, 1024, critic)
        ref = FB.output(FB.exact(p, critic, s, a)[0], critic, HIGH)
        e2 = FB.normwise(model(p, critic, s, a, FB.model_sites(STD, 2)), ref)
        e1 = FB.normwise(model(p, critic, s, a, FB.model_sites(STD, 1)), ref)
        assert FP32_BAR < 0.2 * e2 < e1
