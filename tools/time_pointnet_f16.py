"""Times PointNetVlad(featnet="pointnet") eval at 64 x 4096-point submaps, emb 1024 (--ft: feature_transform=True) in "tf32" and
"f16" precision modes, alternating the two in one process: 3 warm-up steps per mode, then the median of --steps CUDA-event-timed
eager forwards per mode.  A separate ops.profile pass per mode gives the per-call breakdown, and the descriptor error of both modes
is taken against the reference goldens (tests/golden/c1_pointnet_eval.npz, c1_pointnet_ft_eval.npz)."""
import argparse
import statistics
import subprocess
import sys
from collections import defaultdict
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np
import torch
from lpdnet_b200 import ops, synth
from lpdnet_b200.util.PointNetVlad import PointNetVlad

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=30)
ap.add_argument("--batch", type=int, default=64)
ap.add_argument("--ft", action="store_true", help="feature_transform=True (the second, 64 x 64 STN)")
args = ap.parse_args()
assert args.steps >= 20 and torch.cuda.is_available(), "needs a CUDA device and at least 20 timed steps"

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
print(f"GPU: {gpu.strip().splitlines()[0] if gpu.strip() else torch.cuda.get_device_name()}")


def load_model(golden, N, ft):
    g = np.load(ROOT / "tests" / "golden" / f"{golden}.npz", allow_pickle=False)
    shapes = {k: eval(s) for k, s in zip(g["keys"].tolist(), g["shapes"].tolist())}
    m = PointNetVlad(num_points=N, featnet="pointnet", emb_dims=1024, feature_transform=ft)
    m.load_state_dict(synth.fill_state_dict(shapes), strict=True)
    return m.cuda().eval(), g


model, _ = load_model("c1_pointnet_ft_eval" if args.ft else "c1_pointnet_eval", 4096, args.ft)
x = synth.clouds(args.batch, 4096, seed=4321).cuda()
modes = ("tf32", "f16")
print(f"featnet=pointnet, feature_transform={args.ft}, {args.batch} x 4096 points, emb 1024")


def forward(m, mode, inp):
    ops.set_precision(mode)
    with torch.no_grad():
        return m(inp)


for _ in range(3):
    for mode in modes:
        forward(model, mode, x)
torch.cuda.synchronize()
times = {m: [] for m in modes}
for _ in range(args.steps):
    for mode in modes:
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        forward(model, mode, x)
        e.record()
        e.synchronize()
        times[mode].append(s.elapsed_time(e))
med = {m: statistics.median(times[m]) for m in modes}
for m in modes:
    t = sorted(times[m])
    print(f"{m:5s}: median {med[m]:.3f} ms per {args.batch}-submap step (min {t[0]:.3f}, max {t[-1]:.3f}, {args.steps} steps)"
          f" = {args.batch / med[m] * 1e3:.0f} submaps/s")
print(f"f16 / tf32 step time: {med['f16'] / med['tf32']:.3f}")

for mode in modes:
    ops.profile(True)
    forward(model, mode, x)
    rec = ops.profile(False)
    torch.cuda.synchronize()
    per = defaultdict(float)
    for label, s, e in rec:
        per[label] += s.elapsed_time(e)
    total = sum(per.values())
    print(f"\nper-call breakdown, {mode} (profiled pass, event pair around every C-ABI call; sum {total:.3f} ms):")
    for label, ms in sorted(per.items(), key=lambda kv: -kv[1]):
        print(f"  {ms:8.3f} ms  {100 * ms / total:5.1f} %  {label}")

print()
for golden, N, ft in (("c1_pointnet_eval", 4096, False), ("c1_pointnet_ft_eval", 1024, True)):
    m, g = load_model(golden, N, ft)
    xg = synth.clouds(2, N).cuda()
    for mode in modes:
        err = np.abs(forward(m, mode, xg).cpu().numpy() - g["out"]).max()
        print(f"[{mode}] {golden}: max-abs descriptor error vs the reference golden {err:.3e}")
