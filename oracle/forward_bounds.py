"""Per-row error bounds of the actor and critic forward passes (avd_actor_forward / avd_critic_forward), in float64.
TEST INFRASTRUCTURE ONLY.

`exact()` evaluates one network in float64; `row_bound()` gives, for every row, a first-order worst-case bound on
|kernel output - exact()| from the exact intermediates and the operand formats of the path the library runs for (dims,
precision).  `forward_path()` restates csrc/avd_ddpg.cu::fused_path and fused3::supported.

Paths and what they round (u = unit roundoff: bf16 2^-8, fp16 2^-11, fp32 and the three-way split 2^-24):

  fused    precision 1 / 2 when fused3::supported(dims) (avd_fused3.cu): folded formulation
           z1 = s W1 + b1 from hi / lo-split bf16 operands (each factor kept to 2^-16, the lo . lo product dropped:
           3 2^-16 relative to sum |s W1| + |b1|); the critic's action branch fma(a, wa, ba) in fp32;
           r1 = relu(z1) and W2' = diag(sc1) W2 in bf16 (precision 1) or fp16 (precision 2).  Neither fp16 operand is scaled
           (the fused kernel converts r1 with cvt.rn.satfinite.relu.f16x2, pack_fold_kernel converts sc1 W2 with to_op16),
           so below 2^-14 both round in the subnormal range: an absolute floor of 2^-25 per element.
  unfused  precision 0 / 3, and precision 1 / 2 outside fused3::supported: H = BN(relu(z1)) in fp32 (l1_forward_kernel),
           then H and the unfolded W2 in the operand format of csrc/avd_ddpg.cu::operand_format -- fp32 (0), bf16
           (1 AND 2: precision 2 has no fp16 operands on this path) or three bf16 planes (3, 2^-24).

The GEMMs accumulate in fp32: gamma_K = K 2^-24 times the sum of |products|, with K = 2 F to cover the two accumulators
of the split GEMM.  ReLU and tanh are 1-Lipschitz, so a bound on |delta z| carries through them whatever the signs do.
"""
from __future__ import annotations

import numpy as np

F64 = np.float64
BN_EPS = 1e-3
U32 = 2.0 ** -24
U_FMT = {"bf16": 2.0 ** -8, "fp16": 2.0 ** -11, "fp32": U32, "bf16x3": U32}
FP16_FLOOR = 2.0 ** -25        # half the spacing of fp16 subnormals (no power-of-two scale on the forward operands)
FP16_MAX = 65504.0
L1_SPLIT = 3 * 2.0 ** -16      # hi / lo-split layer 1 of the fused kernel, relative to sum |s W1| + |b1|

# csrc/avd_fused3.cu: TILE_M, L2N, L1N, kVRows
FUSED_L1, FUSED_L2, FUSED_LA_MAX = 256, 128, 48


def fused_supported(ns, l1, la, l2):
    """fused3::supported"""
    return l2 == FUSED_L2 and 1 <= ns <= 4 and l1 == FUSED_L1 and la % 16 == 0 and 16 <= la <= FUSED_LA_MAX


def forward_path(dims, precision):
    """'fused' or 'unfused' (csrc/avd_ddpg.cu::fused_path); dims = (ns, l1, la, l2)."""
    return "fused" if precision in (1, 2) and fused_supported(*dims) else "unfused"


def operand_formats(dims, precision):
    """(format of the layer-2 A operand, format of the layer-2 B operand) on the path that runs."""
    if forward_path(dims, precision) == "fused":
        f = "fp16" if precision == 2 else "bf16"
        return f, f
    f = {0: "fp32", 1: "bf16", 2: "bf16", 3: "bf16x3"}[precision]
    return f, f


def model_sites(dims, precision):
    """Rounding sites of tools/precision_model.Net that reproduce the operand formats of the path that runs."""
    fmt = {"fp16": "fp16sat", "bf16": "bf16", "fp32": "fp32", "bf16x3": "bf16x3"}[operand_formats(dims, precision)[0]]
    if forward_path(dims, precision) == "fused":
        return {"l1": "bf16x2", "r1": fmt, "W2f": fmt}
    return {"H": fmt, "W2u": fmt}


def _fold(p, g, be, mu, var):
    sc = p[g] / np.sqrt(p[var] + BN_EPS)
    return sc, p[be] - p[mu] * sc


def exact(p, critic, s, a=None):
    """Float64 forward pass of one network: pre-activation of the head (actor) or q (critic), and the intermediates."""
    p = {k: np.asarray(v, F64) for k, v in p.items()}
    s = np.asarray(s, F64)
    if critic:
        a = np.asarray(a, F64).reshape(-1, 1)
        scs, shs = _fold(p, "gs", "bes", "mus", "vars")
        sca, sha = _fold(p, "ga", "bea", "mua", "vara")
        sc1, sh1 = np.concatenate([scs, sca]), np.concatenate([shs, sha])
        be1, mu1 = np.concatenate([p["bes"], p["bea"]]), np.concatenate([p["mus"], p["mua"]])
        z1 = np.concatenate([s @ p["Ws"] + p["bs"], a @ p["Wa"] + p["ba"]], axis=1)
        l1mag = np.concatenate([np.abs(s) @ np.abs(p["Ws"]) + np.abs(p["bs"]), np.abs(a) @ np.abs(p["Wa"]) + np.abs(p["ba"])], axis=1)
    else:
        sc1, sh1 = _fold(p, "g1", "be1", "mu1", "var1")
        be1, mu1 = p["be1"], p["mu1"]
        z1 = s @ p["W1"] + p["b1"]
        l1mag = np.abs(s) @ np.abs(p["W1"]) + np.abs(p["b1"])
    sc2, sh2 = _fold(p, "g2", "be2", "mu2", "var2")
    w3 = p["W3"][:, 0]
    r1 = np.maximum(z1, 0)
    h1 = r1 * sc1 + sh1
    z2 = h1 @ p["W2"] + p["b2"]
    r2 = np.maximum(z2, 0)
    pre = (r2 * sc2 + sh2) @ w3 + p["b3"][0]
    return pre, dict(p=p, z1=z1, l1mag=l1mag, r1=r1, h1=h1, sc1=sc1, sh1=sh1, be1=be1, mu1=mu1, z2=z2, r2=r2,
                     sc2=sc2, sh2=sh2, w3=w3)


def output(pre, critic, high):
    return pre if critic else high * np.tanh(pre)


def row_bound(p, critic, s, a=None, *, dims, precision, high=2.5):
    """Per-row bound on |kernel output - output(exact())|: the action for the actor, q for the critic.  Rows whose fp16 operands
    would leave the fp16 range (where the kernel saturates) get an infinite bound."""
    pre, c = exact(p, critic, s, a)
    P = c["p"]
    fused = forward_path(dims, precision) == "fused"
    fa, fb = operand_formats(dims, precision)
    ua, ub = U_FMT[fa], U_FMT[fb]
    eta_a = FP16_FLOOR if fa == "fp16" else 0.0
    eta_b = FP16_FLOOR if fb == "fp16" else 0.0
    ns = dims[0]
    r1, sc1, W2 = c["r1"], c["sc1"], P["W2"]
    F = W2.shape[0]
    bnmag1 = np.abs(c["be1"]) + 2 * np.abs(c["mu1"] * sc1)          # what sh1 = be - mu sc is computed from
    if fused:
        dz1 = (L1_SPLIT + 16 * U32) * c["l1mag"]
        A, B = r1, sc1[:, None] * W2
        dA = (1 + ua) * dz1 + ua * np.abs(r1) + eta_a
        dB = (ub + 4 * U32) * np.abs(B) + eta_b
        # b2' = b2 + sum_f sh1 W2 in fp32 (pack_fold_kernel), then added to the accumulator
        dbias = (F + 8) * U32 * (np.abs(P["b2"]) + bnmag1 @ np.abs(W2))
    else:
        dz1 = (ns + 2) * U32 * c["l1mag"]
        A, B = c["h1"], W2
        dH = np.abs(sc1) * dz1 + 6 * U32 * (np.abs(sc1 * r1) + bnmag1)
        dA = dH + ua * (np.abs(A) + dH) + eta_a
        dB = ub * np.abs(B) + eta_b
        dbias = 0.0
    absB = np.abs(B)
    e = dA @ (absB + dB) + np.abs(A) @ dB + 2 * F * U32 * ((np.abs(A) + dA) @ (absB + dB)) + dbias + U32 * np.abs(c["z2"])
    w3p = c["sc2"] * c["w3"]
    l2 = W2.shape[1]
    head = np.abs(c["r2"]) @ np.abs(w3p) + (np.abs(P["be2"]) + 2 * np.abs(P["mu2"] * c["sc2"])) @ np.abs(c["w3"]) + abs(P["b3"][0])
    dpre = e @ (np.abs(w3p) * (1 + 8 * U32)) + (l2 + 16) * U32 * head
    if critic:
        bound = dpre
    else:
        bound = high * dpre + 8 * U32 * high          # tanhf (2 ulp) and the product with high
    if fa == "fp16":
        over = ((np.abs(A) + dA) > FP16_MAX).any(axis=1) | (np.abs(B).max() > FP16_MAX)
        bound = np.where(over, np.inf, bound)
    return bound, output(pre, critic, high)


def normwise(got, ref):
    """max |got - ref| / max |ref| over the rows (the metric of the parity tests)."""
    got, ref = np.asarray(got, F64), np.asarray(ref, F64)
    return float(np.max(np.abs(got - ref)) / max(float(np.max(np.abs(ref))), 1e-30))
