"""C3 training step (2 tuples x 22 clouds x 4096 points, lazy quadruplet loss, lpdnet_b200.optim.Adam) with the DG2 edge tensors in
fp32 ("default") and in fp16 (ops.set_train_precision("f16")), under precision "tf32".

The two modes alternate in one process after a warm-up: each round times one step of each.  Reported per mode: the median step
time over the rounds, the peak of torch.cuda.max_memory_allocated over one step, and a per-kernel breakdown from a separate
ops.profile pass.  Usage: python tools/time_train_f16.py [rounds=30]"""
import statistics
import subprocess
import sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch
from lpdnet_b200 import ops, optim, synth
from lpdnet_b200.loss import pointnetvlad_loss as L
from lpdnet_b200.util.PointNetVlad import PointNetVlad

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 30
assert torch.cuda.is_available(), "time_train_f16.py measures on the GPU"
ops.set_precision("tf32")
Bq, N = 2, 4096
model = PointNetVlad(num_points=N, featnet="lpdnet", emb_dims=1024)
model.load_state_dict(synth.synthetic_state_dict(model))
model = model.cuda().train()
opt = optim.Adam(model.parameters(), lr=1e-3)
x = synth.clouds(Bq * 22, N).cuda()
MODES = ("default", "f16")


def step(mode):
    ops.set_train_precision(mode)
    opt.zero_grad()
    out = model(x)
    q, pos, neg, other = torch.split(out.view(Bq, -1, 256), [1, 2, 18, 1], dim=1)
    loss = L.quadruplet_loss(q, pos, neg, other, 0.5, 0.2, use_min=True, lazy=True)
    loss.backward()
    opt.step()
    return loss


try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                         capture_output=True, text=True).stdout.strip()
except OSError:
    smi = "nvidia-smi not available"
print(f"GPU: {torch.cuda.get_device_name()} ({smi})")

for _ in range(3):
    for m in MODES:
        step(m)
torch.cuda.synchronize()
peak = {}
for m in MODES:
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    step(m)
    torch.cuda.synchronize()
    peak[m] = (torch.cuda.max_memory_allocated(), base)
times = {m: [] for m in MODES}
losses = {}
for _ in range(rounds):
    for m in MODES:
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        loss = step(m)
        e.record()
        e.synchronize()
        times[m].append(s.elapsed_time(e))
        losses[m] = float(loss.detach())
for m in MODES:
    t = times[m]
    print(f"train precision {m:7s}: median {statistics.median(t):.3f} ms/step over {len(t)} steps (min {min(t):.3f}, max {max(t):.3f}); "
          f"peak allocated {peak[m][0] / 2**30:.2f} GiB ({(peak[m][0] - peak[m][1]) / 2**30:.2f} GiB above the resident state); "
          f"last loss {losses[m]:.5f}")
print(f"peak allocated, default - f16: {(peak['default'][0] - peak['f16'][0]) / 2**30:.2f} GiB")

prof = {}
for m in MODES:
    step(m)
    torch.cuda.synchronize()
    ops.profile(True)
    step(m)
    rec = ops.profile(False)
    torch.cuda.synchronize()
    tot = {}
    for label, a, b in rec:
        t = tot.setdefault(label, [0.0, 0])
        t[0] += a.elapsed_time(b)
        t[1] += 1
    prof[m] = tot
    print(f"\n[{m}] sum of profiled calls {sum(v[0] for v in tot.values()):.3f} ms (profiling pass, slower than the timed steps)")
    for k_, v in sorted(tot.items(), key=lambda kv: -kv[1][0])[:30]:
        print(f"  {k_:50s} {v[0]:8.3f} ms  x{v[1]}")
ops.set_train_precision("default")
