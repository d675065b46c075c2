"""What stochastic DDIM costs: CUDA-event milliseconds per plugin forward on BASELINE config 3 (Swin-L, T = 20, 4 x 352 x 1216,
fully native, CUDA graphs, FP8 corrections) at eta = 0 and eta = 1, alternated.  The eta = 1 forward includes the T step
draws (torch.randn on the default CUDA generator), the staging transpose and the sigma * z term of every step.
Prints the card, its power limit and SM clock beside the numbers."""
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import dd_helpers  # noqa: E402
from oracle import restate  # noqa: E402

dev = torch.device("cuda:0")
T, B, H, W = 20, 4, 352, 1216
REPS, ROUNDS = 10, 3
m = dd_helpers.build_mirror("swinl", T).to(dev)
head = m.depth_head
head.check_range = False
s = {k: v.to(dev) for k, v in restate.synthetic_sample(B, H, W).items()}
s["noise"] = restate.synthetic_noise(B, H, W).to(dev)


def timed(eta):
    head.ddim_eta = eta
    with torch.no_grad():
        m(s)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(REPS):
            m(s)
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / REPS


res = {0.0: [], 1.0: []}
for _ in range(ROUNDS):
    for eta in (0.0, 1.0):
        res[eta].append(timed(eta))
smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
t0, t1 = min(res[0.0]), min(res[1.0])
print(f"[clock] {smi}")
print(f"C3 forward, B={B}, T={T}: eta=0 {t0:.2f} ms (rounds {', '.join(f'{v:.2f}' for v in res[0.0])}) | "
      f"eta=1 {t1:.2f} ms (rounds {', '.join(f'{v:.2f}' for v in res[1.0])}) | overhead {t1 - t0:.2f} ms "
      f"({100 * (t1 - t0) / t0:.1f} %)", flush=True)
