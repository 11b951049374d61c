"""Per-tensor error of the tensor-core learn step (precision 1 = bf16 operands, 2 = fp16 operands, 3 = three-way split bf16
operands) against the fp32 oracle, for a few batch sizes.
    python tools/accuracy_report.py [precision ...] > profiles/r03_tensor_core_accuracy.txt      (default: 1 2 3)"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from oracle import ddpg_np as D
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import test_gpu_ddpg as T
from avddpg_b200 import _lib, trainer
from avddpg_b200.config import Config

mods = dict(lib=_lib, trainer=trainer, Config=Config)
print("# rel-L2 error of every gradient tensor, tcgen05 learn step vs oracle/ddpg_np.py (fp32 numpy); seed 50 of tests/test_gpu_ddpg.py")
precisions = [int(x) for x in sys.argv[1:]] or [1, 2, 3]
for prec, R in [(p, R) for p in precisions for R in (64, 1024, 16384, 262144)]:
    conf, pop, nets, batches, (s, a, r, s2) = T.build_population(mods, 1, R, [50])
    pop.precision = prec
    pop.learn(s, a, r, s2, apply_updates=False)
    torch.cuda.synchronize()
    ocg, oag, info = D.learn(nets[0][0], nets[0][1], nets[0][2], nets[0][3], batches[0], gamma=conf.gamma, high=conf.action_high)
    row = []
    for bank, ref in ((pop.critic, ocg), (pop.actor, oag)):
        for name in bank.trainable_names:
            got = bank.view(name, 0, bank.grad).cpu().numpy()
            row.append(f"{bank.kind[0]}.{name}={T._l2(got, ref[name].reshape(got.shape)):.1e}")
    loss = pop.loss[0].cpu().numpy()
    print(f"precision={prec} R={R:7d}  loss_c {abs(loss[0]-info['critic_loss'])/abs(info['critic_loss']):.1e} loss_a {abs(loss[1]-info['actor_loss'])/abs(info['actor_loss']):.1e}  " + " ".join(row))
