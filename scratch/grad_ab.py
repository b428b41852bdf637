"""A/B of gradient-kernel builds at the c5 size: time of the bf16 kernel per 8.4M-sample minibatch (CUDA events, 5 rounds x 4
minibatches after a warm-up round), a hash of the gradient bits of each update precision (fp32, tf32, bf16), the error of the
bf16 kernel against the fp32 CUDA-core kernel.
usage: DRONECU_LIB=path/to/lib.so python scratch/grad_ab.py [n_envs] [K] [minibatches]"""
import sys, os, hashlib, ctypes as C, numpy as np, torch
sys.path.insert(0, '.')
from drone_rl_b200 import _lib
from drone_rl_b200.ppo import PPO
n = int(sys.argv[1]) if len(sys.argv) > 1 else 1048576
K = int(sys.argv[2]) if len(sys.argv) > 2 else 32
mb = int(sys.argv[3]) if len(sys.argv) > 3 else 4
model = PPO(n, n_steps=K, batch_size=n * K // mb, rollout_precision="tf32", update_precision="bf16", seed=3)
model.collect_rollouts()
P = lambda t: None if t is None else C.c_void_p(t.data_ptr())
b, B, m = model.buf, n * K, n * K // mb
perm = torch.empty(B, dtype=torch.int32, device="cuda")
_lib.check(model.lib.dronecu_minibatch_partition(model._h, B, m, 1, 0, P(perm), None))
stats = torch.zeros(mb, 3, dtype=torch.float64, device="cuda")
_lib.check(model.lib.dronecu_ppo_adv_stats_epoch(model._h, P(b.adv), P(perm), B, m, P(stats), None))
g = torch.zeros(_lib.GRAD_LEN, device="cuda")
def launch(k, prec):
    model.launch_grad(perm[k * m:(k + 1) * m], 0, m, P(stats[k]), g, precision=prec)
times = []
for rnd in range(6):
    for k in range(mb):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); launch(k, "bf16"); e1.record(); torch.cuda.synchronize()
        if rnd: times.append(e0.elapsed_time(e1))
hs = {p: hashlib.sha256() for p in ("fp32", "tf32", "bf16")}
errs = []
for k in range(mb):
    gk = {}
    for p, h in hs.items():
        launch(k, p); torch.cuda.synchronize(); gk[p] = g.cpu().numpy().copy()
        h.update(gk[p].tobytes())
    g16, g32 = gk["bf16"][:10697], gk["fp32"][:10697]
    errs.append(float(np.abs(g16 - g32).max() / np.abs(g32).max()))
t = np.array(times)
print(f"{os.environ.get('DRONECU_LIB', 'libdronecu.so'):44s} grad+reduce {t.mean():.4f} ms (min {t.min():.4f}, max {t.max():.4f}) per {m} samples | "
      + " | ".join(f"sha256 {p} {h.hexdigest()[:16]}" for p, h in hs.items())
      + f" | max err vs fp32 / max|g| {max(errs):.2e}", flush=True)
