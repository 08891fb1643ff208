"""Time the feature intensities (BASELINE configs[4] pattern: F = 1024 feature centers, the 14 cuts of
scripts/3_make_rqae_features.py:178, nq = 1024) on synthetic codes resident in HBM; CUDA events.
usage: python tools/bench_intensity.py [--tokens N] [--features F] [--reps R] [--precision tc|exact]

--precision tc (default) times the tcgen05 GEMM and the selection.  --precision exact times both precisions on the
same inputs, after warm-up, and reports ms and (token, feature, layer) elements per second for each; it then checks
|exact - tc| <= 2e-3 on the whole output and the exact path bit for bit against oracle.feature_oracle.intensity_steps
on 16 features x 4096 tokens, and prints the card's name and power limit.  --codes lanes / constant time the exact path on
codes whose look-ups cannot conflict in shared memory (the 32 tokens of a warp read 32 consecutive rows / one row): the
difference to random codes is the cost of bank conflicts."""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from rqae_b200.feature import intensity_many, select_top_middle_bottom

CUTS = [2, 4, 6, 8, 12, 16, 24, 32, 48, 64, 128, 256, 512, 1023]


class Stub:
    quantization_method = "round_fsq"

    def __init__(self, dev):
        from rqae_b200.model import _fsq_grid
        self.codebook = torch.nn.Parameter(_fsq_grid(5, 4, True)[None].to(dev), requires_grad=False)


def _time(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tokens", type=int, default=262144)
    ap.add_argument("--features", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--precision", choices=["tc", "exact"], default="tc")
    ap.add_argument("--codes", choices=["random", "lanes", "constant"], default="random")
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(7)
    codes = torch.randint(0, 625, (a.tokens, 1024), generator=g, device=dev, dtype=torch.int16)
    if a.codes != "random":
        row = torch.arange(a.tokens, device=dev) % 625 if a.codes == "lanes" else torch.zeros(a.tokens, device=dev)
        codes = row.to(torch.int16)[:, None].expand(-1, 1024).contiguous()
    centers = torch.randint(0, 625, (a.features, 1024), generator=g, device=dev, dtype=torch.int32)
    lw = (torch.rand(1024, generator=g, device=dev) * 2 + 13).half()
    m = Stub(dev)
    T_pad = (a.tokens + 255) // 256 * 256
    out = torch.empty(a.features, len(CUTS), T_pad, dtype=torch.float16, device=dev)
    if a.precision == "exact":
        out_x = torch.empty_like(out)
        runs = {"tc": lambda: intensity_many(m, codes, centers, CUTS, layer_weights=lw, out=out),
                "exact": lambda: intensity_many(m, codes, centers, CUTS, layer_weights=lw, out=out_x, precision="exact")}
        for fn in runs.values():
            fn()
        torch.cuda.synchronize()
        elems = a.tokens * a.features * (CUTS[-1] + 1)
        card = _card()
        for name, fn in runs.items():
            ms = _time(fn, a.reps)
            print(json.dumps({"precision": name, "codes": a.codes, "tokens": a.tokens, "features": a.features, "cuts": len(CUTS), "nq": 1024,
                              "ms": ms, "elements_per_s": elems / ms * 1e3, "card": card}))
        worst = 0.0
        for f0 in range(0, a.features, 64):    # whole output, in slices
            d = (out_x[f0:f0 + 64, :, :a.tokens].float() - out[f0:f0 + 64, :, :a.tokens].float()).abs().max()
            worst = max(worst, float(d))
        from oracle import feature_oracle as fo
        sims = fo.codebook_sims(m.codebook.data[0].cpu())
        sub_codes, sub_lw = codes[:4096].cpu(), lw.cpu()
        exact_bits = True
        for f in range(16):
            ref = fo.intensity_steps(sims, centers[f].cpu(), sub_codes, sub_lw, CUTS).T.contiguous()
            exact_bits &= torch.equal(out_x[f, :, :4096].cpu().view(torch.int16), ref.view(torch.int16))
        print(json.dumps({"max_abs_exact_minus_tc": worst, "within_2e-3": worst <= 2e-3,
                          "bit_identical_to_intensity_steps_16x4096": bool(exact_bits), "card": card}))
        if worst > 2e-3 or not exact_bits:
            sys.exit(1)
        return
    for _ in range(2):
        intensity_many(m, codes, centers, CUTS, layer_weights=lw, out=out)
    torch.cuda.synchronize()
    ms = _time(lambda: intensity_many(m, codes, centers, CUTS, layer_weights=lw, out=out), a.reps)
    flop = 2.0 * a.tokens * a.features * 4096
    byts = a.tokens * 2048 + a.features * len(CUTS) * a.tokens * 2
    res = intensity_many(m, codes, centers, CUTS, layer_weights=lw, out=out)
    select_top_middle_bottom(res, 100)
    torch.cuda.synchronize()
    ms_sel = _time(lambda: select_top_middle_bottom(res, 100), a.reps)
    print(json.dumps({"select_ms": ms_sel, "select_gbs": a.features * len(CUTS) * a.tokens * 2 / ms_sel / 1e6,
                      "rows": a.features * len(CUTS)}))
    print(json.dumps({"tokens": a.tokens, "features": a.features, "ms": ms, "tokens_per_s": a.tokens / ms * 1e3,
                      "tflops": flop / ms / 1e9, "out_gbs": byts / ms / 1e6,
                      "note": "whole call: schedule + code transpose + feature operand + GEMM"}))


if __name__ == "__main__":
    main()
