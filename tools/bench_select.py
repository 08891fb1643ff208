"""Timing of the top / middle / bottom selection alone: 14 336 rows x 131 072 fp16 intensities (1024 features x 14 cuts
over one 131 072-token shard), values distributed like intensities (normal around 0, sigma 0.05)."""
import argparse, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from rqae_b200.feature import select_top_middle_bottom

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=14336)
ap.add_argument("--n", type=int, default=131072)
ap.add_argument("--reps", type=int, default=5)
a = ap.parse_args()
dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(3)
v = torch.empty(a.rows, a.n, dtype=torch.float16, device=dev)
for r0 in range(0, a.rows, 1024):
    r1 = min(a.rows, r0 + 1024)
    v[r0:r1] = (0.02 + 0.05 * torch.randn(r1 - r0, a.n, generator=g, device=dev)).half()
idx, val = select_top_middle_bottom(v, 100)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(a.reps):
    idx, val = select_top_middle_bottom(v, 100)
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / a.reps
print(f"select {'v2' if os.environ.get('RQAE_MINE_V2') == '1' else 'v3'}: rows {a.rows} n {a.n}: {ms:.3f} ms, "
      f"{a.rows * a.n * 2 / ms / 1e6:.1f} GB/s of row bytes, checksum {int(idx.long().sum().item())}")
