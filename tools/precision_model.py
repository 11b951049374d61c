"""CPU model of where the tensor-core learn step (precision = 1) loses accuracy against fp32.

Every operand the tcgen05 path rounds is a named SITE; `emulate()` reruns Trainer.learn (workers/trainer.py:489-506) in
float64 with the chosen sites rounded to the chosen format and reports the rel-L2 error of every gradient tensor against the
unrounded run.  Used to decide which operands need more than bf16 (DESIGN.md §4); runs without a GPU:

    python tools/precision_model.py                # table: one site at a time, R = 64 (worst of 20 seeds) and R = 16384
    python tools/precision_model.py --split        # table: every site in one format (fp32, bf16x2, bf16x3, tf32x2), worst
                                                   # per-tensor max-norm error over 40 seeds at R = 64, 4 at 1000, 2 at 16384
                                                   # (the choice of three-way split bf16 operands for precision = 3)

Sites (names follow csrc/avd_fused3.cu / avd_wgrad3.cu / avd_dgrad3.cu):
    l1    state-branch layer 1 of the fused passes: "bf16x2" = the kernel's hi / lo split (s_hi W_hi + s_lo W_hi + s_hi W_lo
          + b_hi + b_lo), "bf16" = hi parts only
    r1    relu(z1) A tile of layer 2, all passes                    W2f   folded layer-2 kernel W2' (forward B operand)
    H     unfused forward: A operand BN(relu(z1))                   W2u   unfused forward: B operand W2 (not folded)
    dm    backward tile dq [z2 > 0] (critic / actor backward)       W2b   W2'' = W2' diag(w3') (dgrad B operand)
    dza   critic-action pass: tile dq w3' [z2 > 0]                  W2a   W2' action rows of the critic-action dgrad
    dz1   staged dz1 chunk (A operand of the layer-1 weight-gradient MMA)
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ddpg_np as D  # noqa: E402

F64 = np.float64
EPS = 1e-3


def rnd(x, fmt):
    if fmt is None:
        return x
    t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
    if fmt == "bf16":
        return t.to(torch.bfloat16).to(torch.float64).numpy()
    if fmt == "fp16":      # per-tensor power-of-two scale so that the largest magnitude sits at 2^14
        m = float(t.abs().max())
        k = 0 if m == 0 else 14 - int(np.ceil(np.log2(m)))
        return (t * 2.0 ** k).to(torch.float16).to(torch.float64).numpy() * 2.0 ** -k
    if fmt == "fp16sat":   # no scale, round to nearest, saturating at +-65504 (the forward pass: pack_fold_kernel, cvt.rn.satfinite)
        return t.clamp(-65504.0, 65504.0).to(torch.float16).to(torch.float64).numpy()
    if fmt == "fp32":      # operands only stored in fp32
        return t.to(torch.float64).numpy()
    if fmt == "bf16x2":    # hi + lo split
        hi = t.to(torch.bfloat16).to(torch.float32)
        lo = (t - hi).to(torch.bfloat16).to(torch.float32)
        return (hi.to(torch.float64) + lo.to(torch.float64)).numpy()
    if fmt == "bf16x3":    # hi + mid + lo split of precision 3 (csrc/avd_ddpg.cu split3), products mid.lo, lo.mid, lo.lo dropped by
        hi = t.to(torch.bfloat16).to(torch.float32)       # the GEMM are below 2^-27 relative and not modelled
        mid = (t - hi).to(torch.bfloat16).to(torch.float32)
        lo = (t - hi - mid).to(torch.bfloat16).to(torch.float32)
        return (hi.to(torch.float64) + mid.to(torch.float64) + lo.to(torch.float64)).numpy()
    if fmt == "tf32x2":    # hi + lo split into 10-bit-significand tf32 (round to nearest on the 13 dropped bits)
        def tf32(v):
            b = v.view(torch.int32)
            return ((b + 0x1000) & ~0x1FFF).view(torch.float32)
        hi = tf32(t.clone())
        lo = tf32((t - hi).contiguous())
        return (hi.to(torch.float64) + lo.to(torch.float64)).numpy()
    raise ValueError(fmt)


def fold(p, g, be, mu, var):
    sc = p[g].astype(F64) / np.sqrt(p[var].astype(F64) + EPS)
    return sc, p[be].astype(F64) - p[mu].astype(F64) * sc


class Net:
    """Folded formulation of one network (critic: state + action branch) with rounding sites."""

    def __init__(self, p, critic, sites):
        self.p, self.critic, self.s = {k: v.astype(F64) for k, v in p.items()}, critic, sites
        p = self.p
        if critic:
            scs, shs = fold(p, "gs", "bes", "mus", "vars")
            sca, sha = fold(p, "ga", "bea", "mua", "vara")
            self.sc1, self.sh1 = np.concatenate([scs, sca]), np.concatenate([shs, sha])
        else:
            self.sc1, self.sh1 = fold(p, "g1", "be1", "mu1", "var1")
        self.sc2, self.sh2 = fold(p, "g2", "be2", "mu2", "var2")
        self.W2p = self.sc1[:, None] * p["W2"]
        self.b2p = p["b2"] + self.sh1 @ p["W2"]
        self.w3p = self.sc2 * p["W3"][:, 0]
        self.b3p = p["b3"][0] + self.sh2 @ p["W3"][:, 0]

    def z1(self, s, a=None):
        p = self.p
        W, b = (p["Ws"], p["bs"]) if self.critic else (p["W1"], p["b1"])
        l1 = self.s.get("l1")
        if l1 is None:
            zs = s @ W + b
        else:                           # hi / lo split of avd_fused3.cu (write_x / W1ext); the lo . lo product is not formed
            hi = lambda x: rnd(x, "bf16")
            sh, Wh, bh = hi(s), hi(W), hi(b)
            zs = sh @ Wh + bh
            if l1 == "bf16x2":
                zs = zs + hi(s - sh) @ Wh + sh @ hi(W - Wh) + hi(b - bh)
            elif l1 != "bf16":
                raise ValueError(l1)
        if self.critic:
            return np.concatenate([zs, a.reshape(-1, 1) @ p["Wa"] + p["ba"]], axis=1)
        return zs

    def forward(self, s, a=None):
        z1 = self.z1(s, a)
        if "H" in self.s:               # unfused forward: BN applied before the rounding, W2 not folded
            h1 = rnd(np.maximum(z1, 0) * self.sc1 + self.sh1, self.s["H"])
            z2 = h1 @ rnd(self.p["W2"], self.s.get("W2u")) + self.p["b2"]
            q = np.maximum(z2, 0) @ self.w3p + self.b3p
            return q, dict(z1=z1, h1=h1, z2=z2)
        r1 = rnd(np.maximum(z1, 0), self.s.get("r1"))
        z2 = r1 @ rnd(self.W2p, self.s.get("W2f")) + self.b2p
        q = np.maximum(z2, 0) @ self.w3p + self.b3p
        return q, dict(z1=z1, r1=r1, z2=z2)

    def backward(self, c, dq, s, a=None):
        """Gradients of the Keras trainable tensors from dq[n] (the unfold of csrc/avd_ddpg.cu::unfold_kernel)."""
        p, S = self.p, self.s
        m2 = (c["z2"] > 0).astype(F64)
        dm = rnd(dq[:, None] * m2, S.get("dm"))
        G2m = c["r1"].T @ dm                                  # wgrad3: recomputed r1 (same rounding) x dm
        dbm = dm.sum(0)
        W2pp = rnd(self.W2p * self.w3p[None, :], S.get("W2b"))
        dR = dm @ W2pp.T                                      # dgrad3
        dz1 = rnd(dR * (c["z1"] > 0), S.get("dz1"))
        g = {}
        G2, db2 = G2m * self.w3p[None, :], self.w3p * dbm
        g["W2"] = self.sc1[:, None] * G2 + self.sh1[:, None] * db2[None, :]
        g["b2"] = db2
        dsh1 = p["W2"] @ db2
        dsc1 = (p["W2"] * G2).sum(1)
        U = (rnd(self.W2p, S.get("W2f")) * G2m).sum(0) + self.b2p * dbm
        sd = dq.sum()
        inv2 = 1 / np.sqrt(p["var2"] + EPS)
        g["W3"] = (self.sc2 * U + self.sh2 * sd)[:, None]
        g["g2"] = p["W3"][:, 0] * inv2 * (U - p["mu2"] * sd)
        g["be2"] = p["W3"][:, 0] * sd
        g["b3"] = np.array([sd])
        if self.critic:
            l1 = p["Ws"].shape[1]
            invs, inva = 1 / np.sqrt(p["vars"] + EPS), 1 / np.sqrt(p["vara"] + EPS)
            g["bes"], g["bea"] = dsh1[:l1], dsh1[l1:]
            g["gs"] = invs * (dsc1[:l1] - p["mus"] * dsh1[:l1])
            g["ga"] = inva * (dsc1[l1:] - p["mua"] * dsh1[l1:])
            g["Ws"], g["bs"] = s.T @ dz1[:, :l1], dz1[:, :l1].sum(0)
            g["Wa"], g["ba"] = a.reshape(1, -1) @ dz1[:, l1:], dz1[:, l1:].sum(0)
        else:
            inv1 = 1 / np.sqrt(p["var1"] + EPS)
            g["be1"] = dsh1
            g["g1"] = inv1 * (dsc1 - p["mu1"] * dsh1)
            g["W1"], g["b1"] = s.T @ dz1, dz1.sum(0)
        return g

    def action_grad(self, c, dq_const, a):
        """d(-mean q)/d action per row: the critic-action pass."""
        p, S = self.p, self.s
        l1 = p["Ws"].shape[1]
        m2 = (c["z2"] > 0).astype(F64)
        if S.get("action_T"):          # proposed: A = [z2 > 0] (exact), B = T = W2'[action rows] diag(w3') in the given format
            T = rnd(self.W2p[l1:] * self.w3p[None, :], S["action_T"])
            dRa = dq_const * (m2 @ T.T)
        else:                           # round 1: A = bf16(dq w3' [z2 > 0]), B = bf16 W2'[action rows]
            dza = rnd(dq_const * self.w3p[None, :] * m2, S.get("dza"))
            dRa = dza @ rnd(self.W2p[l1:], S.get("W2a")).T
        za = c["z1"][:, l1:]
        return ((za > 0) * dRa) @ p["Wa"][0]


def emulate(nets, batch, sites, gamma=0.99, high=2.5):
    actor, critic, t_actor, t_critic = nets
    s, a, r, s2 = (np.asarray(x, F64) for x in batch)
    a, r = a.reshape(-1), r.reshape(-1)
    R = len(s)
    TA, TC, Cr, Ac = Net(t_actor, False, sites), Net(t_critic, True, sites), Net(critic, True, sites), Net(actor, False, sites)
    a2 = high * np.tanh(TA.forward(s2)[0])
    y = r + gamma * TC.forward(s2, a2)[0]
    q, cc = Cr.forward(s, a)
    cg = Cr.backward(cc, 2 * (q - y) / R, s, a)
    pre, ca = Ac.forward(s)
    pi = high * np.tanh(pre)
    _, cc2 = Cr.forward(s, pi)
    dpi = Cr.action_grad(cc2, -1.0 / R, pi)
    ag = Ac.backward(ca, dpi * high * (1 - np.tanh(pre) ** 2), s)
    return cg, ag


def make_case(seed, R):
    rng = np.random.default_rng(seed)
    nets = [D.init_actor(rng), D.init_critic(rng), D.init_actor(rng), D.init_critic(rng)]
    for n, crit in zip(nets, (False, True, False, True)):
        D.randomize_bn(n, rng, [("gs", "bes", "mus", "vars"), ("ga", "bea", "mua", "vara"), ("g2", "be2", "mu2", "var2")] if crit
                       else [("g1", "be1", "mu1", "var1"), ("g2", "be2", "mu2", "var2")])
    nets = [nets[0], nets[1], nets[2], nets[3]]
    sb = rng.normal(0, 2, (R, 4)).astype(np.float32)
    batch = (sb, rng.uniform(-2.5, 2.5, (R, 1)).astype(np.float32), -rng.uniform(0, 0.5, (R, 1)).astype(np.float32),
             (sb + rng.normal(0, 0.2, (R, 4))).astype(np.float32))
    return (nets[0], nets[1], nets[2], nets[3]), batch


def errors(ref, got):
    out = {}
    for (rc, ra), (gc, ga), tag in ((ref, got, ""),):
        for k in rc:
            out["c." + k] = float(np.linalg.norm(gc[k].ravel() - rc[k].ravel()) / max(np.linalg.norm(rc[k].ravel()), 1e-300))
        for k in ra:
            out["a." + k] = float(np.linalg.norm(ga[k].ravel() - ra[k].ravel()) / max(np.linalg.norm(ra[k].ravel()), 1e-300))
    return out


ROUND1 = dict(r1="bf16", W2f="bf16", dm="bf16", W2b="bf16", dza="bf16", W2a="bf16", dz1="bf16")


def report(configs, Rs=(64, 16384), seeds64=20):
    for name, sites in configs:
        for R in Rs:
            worst = {}
            for seed in range(seeds64 if R <= 256 else 2):
                nets, batch = make_case(100 + seed, R)
                e = errors(emulate(nets, batch, {}), emulate(nets, batch, sites))
                for k, v in e.items():
                    worst[k] = max(worst.get(k, 0.0), v)
            cmax = max(v for k, v in worst.items() if k.startswith("c."))
            amax = max(v for k, v in worst.items() if k.startswith("a."))
            keys = ["c.Ws", "c.W2", "c.W3", "a.W1", "a.W2", "a.b3"]
            print(f"{name:34s} R={R:6d} critic max {cmax:.1e} actor max {amax:.1e}  " + " ".join(f"{k}={worst[k]:.1e}" for k in keys), flush=True)


SPLIT_SITES = ("r1", "W2f", "dm", "W2b", "dz1", "action_T")


def report_split(fmts=("fp32", "bf16x2", "bf16x3", "tf32x2"), cases=((64, 40), (1000, 4), (16384, 2))):
    """Every rounding site in one format; worst per-tensor max-norm error (max |got - ref| / max |ref|, the metric of the
    precision-0 parity test) against the unrounded float64 run, over the seeds of each batch size."""
    for fmt in fmts:
        sites = {k: fmt for k in SPLIT_SITES}
        row = []
        for R, nseeds in cases:
            worst, where = 0.0, None
            for seed in range(nseeds):
                nets, batch = make_case(100 + seed, R)
                for (rc, ra), (gc, ga) in ((emulate(nets, batch, {}), emulate(nets, batch, sites)),):
                    for tag, ref, got in (("c.", rc, gc), ("a.", ra, ga)):
                        for k in ref:
                            e = float(np.max(np.abs(got[k] - ref[k])) / max(np.max(np.abs(ref[k])), 1e-300))
                            if e > worst:
                                worst, where = e, f"{tag}{k} seed {seed}"
            row.append(f"R={R:6d} ({nseeds:2d} seeds) {worst:.1e} [{where}]")
        print(f"{fmt:7s} " + "  ".join(row), flush=True)


if __name__ == "__main__":
    if "--split" in sys.argv:
        report_split()
        sys.exit(0)
    one_at_a_time = [("round 1 (all bf16)", ROUND1)] + [(f"only {k}", {k: "bf16"}) for k in ("r1", "W2f", "dm", "W2b", "dz1")] + [
        ("only dza+W2a (critic-action)", {"dza": "bf16", "W2a": "bf16"})]
    report(one_at_a_time)
