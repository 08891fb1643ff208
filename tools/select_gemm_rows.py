"""Selection on the intensity GEMM's own rows, cut by cut: time of the sample-bracketed kernel and of the three-pass
kernel.  usage: python tools/select_gemm_rows.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from rqae_b200 import RQAE
from rqae_b200.feature import intensity_many, select_top_middle_bottom, layer_weights_f16

CUTS = [2, 4, 6, 8, 12, 16, 24, 32, 48, 64, 128, 256, 512, 1023]   # scripts/3_make_rqae_features.py:178
dev = torch.device("cuda:0")
torch.manual_seed(0)
model = RQAE(dim=2304, num_quantizers=1024).eval().to(dev)
T, Fn = 131072, 1024
x = torch.randn(T, 2304, device=dev, generator=torch.Generator(device=dev).manual_seed(5))
codes = model.encode(x, out_dtype=torch.int16)
codes = codes.reshape(T, -1)
centers = codes[torch.randperm(T, device=dev)[:Fn]].to(torch.int32)
lw = layer_weights_f16(model).to(dev)
out = intensity_many(model, codes, centers, CUTS, layer_weights=lw)
torch.cuda.synchronize()
print("rows", tuple(out.shape), "distinct values in row 0 per cut:", [int(out[0, c].unique().numel()) for c in range(len(CUTS))])


def ms(fn, reps=2):
    fn(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


for c, cut in enumerate(CUTS):
    rows = out[:, c, :]
    sys.stderr.flush()
    print(f"cut {cut}:", flush=True)
    t3 = ms(lambda: select_top_middle_bottom(rows, 100), reps=1)
    os.environ["RQAE_MINE_V2"] = "1"
    t2 = ms(lambda: select_top_middle_bottom(rows, 100), reps=1)
    os.environ.pop("RQAE_MINE_V2")
    print(f"   v3 {t3:.3f} ms   v2 {t2:.3f} ms", flush=True)
