#!/usr/bin/env python
"""bench.py -- throughput of the RQAE residual-quantization hot path (forward = encode + reconstruction).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--tokens T] [--dump-outputs DIR]

One "step" = one pass of RQAE.forward over T synthetic N(0,1) activation tokens per GPU at Gemma-2-2B
width (d=2304, nq=1024, K=625, random init from torch.manual_seed(0)): BASELINE.json configs[1].
`value` is whole-job tokens/s with the inputs resident in HBM (CUDA events, max over ranks);
`e2e` is the same metric through RQAE.forward_host with pinned HOST buffers (H2D of the activations
and D2H of codes + reconstruction inside the timed region).  N>1: one process per GPU (torchrun), every
rank processes its own T tokens (weak scaling), no collective on the data path.

`--impl reference` times the reference's CPU implementation of the same path on the host cores: the
unmodified /root/reference module when it exists (build container), else the op-for-op torch port in
oracle/rqae_oracle.py (the GPU box has no /root/reference).

`--dump-outputs DIR` writes what RQAE.forward returned in the last timed step (rank 0's tokens) as
DIR/quantized_out.npy (float32) and DIR/indices.npy (float64, exact for the int64 codes), at the same seeded sample
of token rows on every run, so that two builds given the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

D, NQ, K_ROWS = 2304, 1024, 625
FLOP_PER_TOKEN_FWD = NQ * 46472          # SURVEY 8d: 2*4*D in-proj + 2*4*K cos + 2*4*D out-proj + D + D
HBM_BYTES_PER_TOKEN_FWD = 4 * D + 8 * NQ + 4 * D   # x in, int64 codes out, fp32 reconstruction out
METRIC = "rq_forward_encode_decode_tokens_per_sec"
UNIT = "tokens/s"
DUMP_ROWS = 3072    # token rows of --dump-outputs: 3072 x (2304 x 4 B + 1024 x 8 B) = 53.5 MB, within 64 MB


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--tokens", type=int, default=1 << 20, help="tokens per GPU per step")
    ap.add_argument("--e2e-tokens", type=int, default=0, help="tokens per e2e step (default: --tokens)")
    ap.add_argument("--e2e-steps", type=int, default=0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU work per reference step")
    ap.add_argument("--no-extras", action="store_true", help="skip the side measurements (mining stage, 9B encode)")
    ap.add_argument("--no-parity", action="store_true", help="skip the 4096-token KAT parity block")
    ap.add_argument("--tokens-9b", type=int, default=1 << 20, help="tokens per GPU of the configs[3] extra")
    ap.add_argument("--tokens-mining", type=int, default=1 << 21, help="tokens per GPU of the configs[4] extra")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs (a fixed sample of %d token rows) as DIR/<name>.npy"
                         % DUMP_ROWS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


# ----------------------------------------------------------------------------------------------------
# CPU arm (reference / port)
# ----------------------------------------------------------------------------------------------------
class CpuArm:
    """The reference's own forward on host cores.  kind = "reference" when /root/reference is importable
    (unmodified rqae.model.RQAE), else "port" (oracle/rqae_oracle.py: same ATen ops in the same order)."""

    def __init__(self):
        import torch
        self.torch = torch
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        self.kind = "port"
        self.fn = None
        if os.path.isdir("/root/reference/rqae"):
            try:
                sys.path.insert(0, "/root/reference")
                from rqae.model import RQAE as Ref
                torch.manual_seed(0)
                ref = Ref().eval()
                self.fn = lambda x: ref(x)
                self.kind = "reference"
            except Exception:
                self.fn = None
        if self.fn is None:
            from oracle import rqae_oracle as orc
            w = orc.random_init()  # same parameter stream as torch.manual_seed(0); RQAE()
            self.fn = lambda x: orc.forward(w, x)

    def run(self, n_tokens: int, seed: int = 1):
        torch = self.torch
        x = torch.randn(1, n_tokens, D, generator=torch.Generator().manual_seed(seed))
        t0 = time.perf_counter()
        with torch.inference_mode():
            self.fn(x)
        return time.perf_counter() - t0

    def calibrate(self, target_s: float) -> int:
        self.run(32)            # first call pays thread-pool and allocator warm-up
        t = self.run(96)
        rate = 96 / t
        n = int(max(32, min(4096, rate * target_s)))
        return (n + 31) // 32 * 32


def cpu_baseline(target_s: float):
    arm = CpuArm()
    n = arm.calibrate(target_s)
    t = arm.run(n)
    return {"value": n / t, "unit": UNIT, "cores": arm.cores, "kind": arm.kind,
            "sample": f"{n} of the workload's tokens, full depth (nq={NQ}), torch CPU fp32, {t:.1f} s"}


def run_reference(args, rank):
    if rank != 0:
        return
    arm = CpuArm()
    n = arm.calibrate(args.cpu_seconds)
    for _ in range(args.warmup):
        arm.run(max(32, n // 8))
    t = 0.0
    for s in range(args.steps):
        t += arm.run(n, seed=1 + s)
    v = n * args.steps / t
    out = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE configs[1]: random-init RQAE d=2304 nq=1024 K=625, forward "
                               "(encode + reconstruction) of synthetic N(0,1) tokens",
                   "tokens_per_step": n, "note": "bounded sample of the 1Mi-token workload on the host cores"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": arm.cores, "kind": arm.kind,
                         "sample": f"{n} tokens/step, full depth, torch CPU fp32, all host threads"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# ----------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.proc = None
        self.path = f"/tmp/rqae_clocks_{os.getpid()}.csv"
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            p = [s.strip() for s in line.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1])); pw.append(float(p[2]))
            except ValueError:
                continue
            for nme, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------------
def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


def fp32_peak_tflops(torch, lib, dev):
    """Live FP32-pipe peak: the library's FFMA2 / FFMA probe kernels, CUDA events, best of 5."""
    import ctypes
    sink = torch.rand(256, device=dev) + 0.5
    best = {}
    for packed in (1, 0, 2, 3):
        flops = ctypes.c_double(0)
        st = torch.cuda.current_stream(dev).cuda_stream
        name = {1: "ffma2", 0: "ffma", 2: "pattern_inproj", 3: "pattern_outproj"}[packed]
        lib.rqae_fp32_peak_probe(packed, 2000, ctypes.byref(flops), sink.data_ptr(), st)  # warm-up
        torch.cuda.synchronize(dev)
        b = 0.0
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            lib.rqae_fp32_peak_probe(packed, 200000 if packed >= 2 else 20000, ctypes.byref(flops), sink.data_ptr(), st)
            e1.record()
            torch.cuda.synchronize(dev)
            b = max(b, flops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        best[name] = b
    return best


SCRIPT3_CUTS = [2, 4, 6, 8, 12, 16, 24, 32, 48, 64, 128, 256, 512, 1023]   # scripts/3_make_rqae_features.py:178


def _event_ms(torch, dev, fn, reps=2):
    fn(); torch.cuda.synchronize(dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = fn()
    b.record(); torch.cuda.synchronize(dev)
    return out, a.elapsed_time(b) / reps


def mining_extras(torch, model, codes, dev):
    """BASELINE configs[4] pattern on this GPU's own codes: intensities of F = 1024 feature centers (codes of 1024
    tokens) at the 14 cuts of scripts/3 over the token shard (tcgen05 GEMM), then the top / middle / bottom-100
    selection per (feature, cut).  Side measurement, CUDA events, outside the timed region."""
    from rqae_b200.feature import intensity_many, select_top_middle_bottom, layer_weights_f16
    T = codes.shape[0]
    Fn = 1024
    centers = codes[torch.randperm(T, device=dev)[:Fn]].to(torch.int32)
    lw = layer_weights_f16(model).to(dev)
    buf = torch.empty(Fn, len(SCRIPT3_CUTS), (T + 255) // 256 * 256, dtype=torch.float16, device=dev)
    out, ms_int = _event_ms(torch, dev, lambda: intensity_many(model, codes, centers, SCRIPT3_CUTS, layer_weights=lw, out=buf))
    (idx, val), ms_sel = _event_ms(torch, dev, lambda: select_top_middle_bottom(out, 100))
    # the same rows through the three-pass kernel (the sample-bracketed kernel's fallback), for the A/B
    os.environ["RQAE_MINE_V2"] = "1"
    try:
        (idx2, _), ms_sel2 = _event_ms(torch, dev, lambda: select_top_middle_bottom(out, 100))
    finally:
        os.environ.pop("RQAE_MINE_V2", None)
    assert torch.equal(idx, idx2), "selection: the single-pass kernel and the three-pass kernel disagree"
    peaks = measured_peaks()
    tensor_peak = peaks["bf16_tflops"] if peaks else 1590.0
    hbm_peak = peaks["hbm_gbs"] if peaks else 6650.0
    flop = 2.0 * T * Fn * 4 * (SCRIPT3_CUTS[-1] + 1)
    out_bytes = Fn * len(SCRIPT3_CUTS) * T * 2
    res = {
        "tokens": T, "features": Fn, "cuts": len(SCRIPT3_CUTS),
        "intensity_ms": ms_int, "intensity_tokens_per_s": T / ms_int * 1e3,
        "intensity_tflops": flop / ms_int / 1e9, "intensity_frac_of_tensor_peak": flop / ms_int / 1e9 / tensor_peak,
        "intensity_out_gbs": out_bytes / ms_int / 1e6, "intensity_frac_of_hbm_peak": out_bytes / ms_int / 1e6 / hbm_peak,
        "tensor_peak_source": "MEASURED_PEAKS.json (burst)" if peaks else "fallback 1.59 PFLOP/s (B200_PROFILING.md)",
        "select_ms": ms_sel, "select_rows_per_s": Fn * len(SCRIPT3_CUTS) / ms_sel * 1e3,
        "select_gbs": out_bytes / ms_sel / 1e6, "select_frac_of_hbm_peak": out_bytes / ms_sel / 1e6 / hbm_peak,
        "select_kernel": "rq_mine3 (brackets from a 1/16 sample, one streaming pass; rows whose brackets miss go to rq_mine2)",
        "select_ms_three_pass_kernel": ms_sel2, "select_equal_to_three_pass_kernel": True,
        "checksum_top_idx": int(idx[:, :, 0].sum().item()),
    }
    # the reference's CPU path for the same step (one feature at a time, rqae/feature.py:102-129), bounded sample
    try:
        from oracle import feature_oracle as fo
        import time as _t
        n = min(T, 16384)
        cc = codes[:n].cpu().long()
        sims = fo.codebook_sims(model.codebook.data[0].cpu())
        c0 = centers[0].cpu()
        lwc = lw.cpu()
        fo.intensity(sims, c0, cc[:256], lwc, SCRIPT3_CUTS)
        t0 = _t.perf_counter()
        v = fo.intensity(sims, c0, cc, lwc, SCRIPT3_CUTS)
        t1 = _t.perf_counter()
        for j in range(len(SCRIPT3_CUTS)):
            fo.select_top_middle_bottom(v[:, j], 100)
        t2 = _t.perf_counter()
        res["cpu_port"] = {"feature_tokens_per_s_intensity": n / (t1 - t0), "feature_tokens_per_s_select": n / (t2 - t1),
                           "gpu_feature_tokens_per_s_intensity": T * Fn / ms_int * 1e3,
                           "sample": f"1 feature x {n} tokens x {len(SCRIPT3_CUTS)} cuts, torch CPU (oracle port of feature.py)"}
    except Exception as e:
        res["cpu_port"] = {"error": repr(e)}
    return res


def search_cpu_port(torch, sims_cpu, sequences=256, positions=127, seed=78):
    """The reference's CPU path for the example search (oracle port of demo/server/server.py:159-325, same ATen calls),
    on a bounded sample of the store: `sequences` synthetic sequences, one 127-position query, the server's 13 cuts."""
    from oracle import search_oracle as so
    import time as _t
    nq, K = sims_cpu.shape[0], sims_cpu.shape[1]
    g = torch.Generator().manual_seed(seed)
    codes = torch.randint(0, K, (sequences, positions, nq), generator=g, dtype=torch.int32)
    k = min(10, sequences)
    t0 = _t.perf_counter()
    n = 0
    for _res, _layer in so.find_examples([codes], sims_cpu, codes[sequences // 3], k, k, k, so.SERVER_LAYERS):
        n += 1
    dt = _t.perf_counter() - t0
    return {"sequences_per_s": sequences / dt, "seconds": dt, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{sequences} sequences x {positions} positions x {max(so.SERVER_LAYERS)} layers, 127-position query, "
                      f"{n} cuts, torch CPU (oracle port of server.py find_examples)"}


def search_extras(torch, model, dev, sequences=36864, positions=127):
    """SURVEY 8f-3: nearest-example search (demo/server/server.py:159-325) over a code store of the reference's shape
    (36 864 sequences x 127 positions x 1024 layers, server.py:139; synthetic uniform codes, int16, resident in HBM) with
    the engine table of THIS model (subfeature_sims * layer_norms), one 127-position query, the server's 13 layer cuts,
    top-30 / middle-10 / bottom-10 after every cut.  Side measurement, CUDA events, outside the timed region."""
    from rqae_b200 import _lib
    from rqae_b200.search import IntensityEngine, SERVER_LAYERS, engine_sims
    nq, K = model.num_quantizers, model.codebook.shape[1]
    g = torch.Generator(device=dev).manual_seed(77)
    codes = torch.randint(0, K, (sequences, positions, nq), generator=g, device=dev, dtype=torch.int16)
    eng = IntensityEngine(sims=engine_sims(model), activations=codes)
    lib = _lib.load()
    idx = sequences // 3

    def one():
        last = None
        for res, layer in eng.find_examples(idx=idx):
            last = res
        return last
    n0 = int(lib.rqae_launch_count(0))
    res, ms = _event_ms(torch, dev, one, reps=2)                   # one warm-up pass + two timed
    launches = (int(lib.rqae_launch_count(0)) - n0) // 3
    L = max(SERVER_LAYERS)
    rows = sequences * positions * L
    peaks = measured_peaks()
    hbm_peak = peaks["hbm_gbs"] if peaks else 6650.0
    # algorithmic HBM bytes: the code store once + the fp16 accumulation written once per cut and re-read by the next cut
    # and by the per-position max
    acc_bytes = sequences * positions * 128 * 2
    hbm = rows * 2 + acc_bytes * (3 * len(SERVER_LAYERS) - 1)
    try:
        cpu = search_cpu_port(torch, eng.sims.cpu())
    except Exception as e:
        cpu = {"error": repr(e)}
    # opt-in tensor-core ranking (precision="tc"): one GEMM launch for the maxima of all cuts + exact rows of the selected
    tc = {}
    try:
        del eng
        eng_tc = IntensityEngine(model, codes, precision="tc")
        query = eng_tc._query(idx, None, L)

        def one_tc():
            last = None
            for r, layer in eng_tc.find_examples(idx=idx):
                last = r
            return last
        res_tc, ms_tc = _event_ms(torch, dev, one_tc, reps=2)
        _, ms_max = _event_ms(torch, dev, lambda: eng_tc.maxima_tc(query, SERVER_LAYERS), reps=2)
        # algorithmic: the code store once (2 B per token-layer); on-chip, one 16-byte factor row per token-layer from L2
        tc = {"find_examples_ms": ms_tc, "sequences_per_s": sequences / ms_tc * 1e3, "maxima_gemm_ms": ms_max,
              "gemm_tflops": 2.0 * rows * 8 * 128 / ms_max / 1e9, "factor_row_tbps": rows * 16 / ms_max / 1e9,
              "hbm_gbs": rows * 2 / ms_max / 1e6, "hbm_frac_of_peak": rows * 2 / ms_max / 1e6 / hbm_peak,
              "self_match_top1": bool((res_tc["top"]["indices"][:, 0] == idx).all().item()),
              "top_overlap_with_exact_last_cut": float((res_tc["top"]["indices"].unsqueeze(2) == res["top"]["indices"].unsqueeze(1))
                                                       .any(dim=2).float().mean().item()),
              "note": "ranking from the rank-5 tensor-core GEMM (maxima within a few fp16 steps of the exact mode, "
                      "tests/test_search_gpu.py); reported intensities recomputed exactly for the selected sequences"}
        del eng_tc
    except Exception as e:
        tc = {"error": repr(e)}
    return {
        "cpu_port": cpu, "tensor_core_ranking_opt_in": tc,
        "sequences": sequences, "positions": positions, "layers": L, "query_positions": positions, "cuts": len(SERVER_LAYERS),
        "find_examples_ms": ms, "sequences_per_s": sequences / ms * 1e3, "launches_per_query": launches,
        "table_row_tbps": rows * 256 / ms / 1e9, "hbm_gbs": hbm / ms / 1e6, "hbm_frac_of_peak": hbm / ms / 1e6 / hbm_peak,
        "bound": "L2 -> SM delivery of 256-byte table rows (DESIGN.md 4.6); HBM fraction shown for scale",
        "self_match_top1": bool((res["top"]["indices"][:, 0] == idx).all().item()),
        "includes": "query table build, 13 x (accumulate + per-position max + radix select), gather of the selected rows and "
                    "their device->host copies (the reference's .cpu() calls)",
    }


def parity_block(torch, model, dev):
    """BASELINE configs[0] through the SAME model object that is timed below: the 4096 KAT tokens
    (torch.manual_seed(0) weights, x = randn(32,128,2304) from CPU seed 1) against the codes of the unmodified
    reference (tests/golden/kat_2b_codes4096.npz) under the near-tie protocol of SURVEY 8c (tests/parity.py):
    a token whose first differing layer has an fp64 margin (teacher-forced along the reference's trajectory,
    C oracle) below eps is a near-tie flip, anything else a failure."""
    import hashlib
    import numpy as np
    from oracle import c_oracle
    from oracle import rqae_oracle as orc
    from tests import parity
    gdir = os.path.join(ROOT, "tests", "golden")
    g = np.load(os.path.join(gdir, "kat_2b.npz"))
    ref = np.load(os.path.join(gdir, "kat_2b_codes4096.npz"))["codes4096"]
    x = torch.randn(32, 128, D, generator=torch.Generator().manual_seed(1))
    if hashlib.sha256(x.numpy().tobytes()).hexdigest()[:16] != str(g["fp_x"]):
        return {"error": "KAT input does not reproduce on this torch build"}
    q, codes = model(x.to(dev))
    codes = codes.cpu().numpy().reshape(4096, NQ)
    q = q.cpu().numpy().reshape(4096, D)
    bad = np.flatnonzero((codes != ref).any(axis=1))
    margins = np.full(ref.shape, np.inf, np.float32)
    if len(bad):
        w = orc.StackedWeights.from_state_dict({k: v.detach().cpu() for k, v in model.state_dict().items()})
        cw = c_oracle.CWeights.from_stacked(w)
        _, _, mb = c_oracle.forward_f64(cw, x.view(-1, D).numpy()[bad], teacher=ref[bad])
        margins[bad] = mb
    rep = parity.compare_codes(codes, ref, margins)
    ok128 = parity.exact_token_mask(codes[:128], ref[:128])
    rel = float(np.abs(q[:128][ok128] - g["q128"][ok128]).max() / np.abs(g["q128"]).max())
    flips = [{"token": int(t), "layer": int(np.argmax(codes[t] != ref[t])),
              "fp64_margin": float(margins[t, int(np.argmax(codes[t] != ref[t]))])} for t in bad[:32]]
    return {"tokens": rep.tokens, "exact": rep.exact, "near_tie": rep.near_tie, "failures": rep.failures,
            "eps": parity.EPS, "worst_accepted_margin": rep.worst_margin, "flips": flips,
            "recon_max_rel_err_first128": rel, "recon_tolerance": 2e-5,
            "reference": "unmodified rqae.model.RQAE on BASELINE configs[0] (tests/golden/kat_2b_codes4096.npz, "
                         "sha %s); margins: fp64 C oracle teacher-forced along the reference's codes" % str(g["fp_codes_i16"])}


class GemmaStub:
    """The two methods RQAE.hook needs from rqae/llm.py:65-73 (Gemma2.norm = the model's final RMSNorm,
    x * rsqrt(mean(x^2) + eps) * (1 + w); denorm inverts it) with a synthetic norm weight."""

    def __init__(self, torch, dim, dev, eps=1e-6):
        self.torch = torch
        self.eps = eps
        self.weight = (0.1 * torch.randn(dim, generator=torch.Generator().manual_seed(5))).to(dev)
        self.rms_weight, self.rms_eps = self.weight, eps      # what the fused hook path reads

    def norm(self, hs):
        t = self.torch
        x = hs.float()
        return (x * t.rsqrt(x.pow(2).mean(-1, keepdim=True) + self.eps) * (1.0 + self.weight.float())).type_as(hs)

    def denorm(self, hs, orig):
        t = self.torch
        hs = hs / (1.0 + self.weight.float())
        return hs.float() / t.rsqrt(orig.float().pow(2).mean(-1, keepdim=True) + 1e-6)


def hook_extra(torch, model, dev, batch=4, seq=128, reps=20):
    """The production caller's operating point (scripts/1_create_activations.py:152: 4 sequences x 128 tokens of
    fp16 hidden states through hook_fn, model.py:276-289): microseconds per hook call, generic path (torch
    norm / denorm around the fused layer loop) and fused path (one launch), CUDA events."""
    stub = GemmaStub(torch, D, dev)
    hs = (3.0 * torch.randn(batch, seq, D, generator=torch.Generator().manual_seed(6))).to(dev).half()
    out = {"batch": batch, "seq": seq, "tokens": batch * seq, "dtype": "fp16"}
    results = {}
    for name, kw in (("generic", dict(norm=stub.norm, denorm=stub.denorm, fused=False)),
                     ("fused", dict(norm=stub.norm, denorm=stub.denorm, rms_weight=stub.rms_weight, rms_eps=stub.rms_eps))):
        try:
            fn = model.hook(**kw)
        except TypeError:
            continue
        buf = hs.clone()
        fn(None, None, (buf,))
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            buf.copy_(hs)
            fn(None, None, (buf,))
        b.record()
        torch.cuda.synchronize(dev)
        results[name] = buf.float()
        out[name + "_us_per_call"] = a.elapsed_time(b) / reps * 1e3
        out[name + "_tokens_per_s"] = batch * seq / (a.elapsed_time(b) / reps * 1e-3)
    if "generic" in results and "fused" in results:
        d = (results["generic"] - results["fused"]).abs()
        tok_same = (d.amax(-1) <= 2e-3 * results["generic"].abs().amax()).float().mean().item()
        out["fused_vs_generic_tokens_within_fp16_rounding"] = tok_same
    return out


def stock_pytorch_gpu_extra(torch, model, dev, sizes=(512, 4096, 65536)):
    """The bar on the same box (SURVEY 2.1 / 8d, BASELINE.md 4.5): the reference's own ATen op sequence with the
    weights on the GPU (what scripts/1:144 does with .to("cuda"); the op-for-op port, ~13 launches per layer) next
    to this repo's fused kernel on the same tokens.  tokens/s for forward (encode + reconstruction)."""
    from oracle import rqae_oracle as orc
    w = orc.StackedWeights.from_state_dict({k: v.detach() for k, v in model.state_dict().items()}).to(dev)
    res = {}
    for n in sizes:
        x = torch.randn(1, n, D, device=dev, generator=torch.Generator(device=dev).manual_seed(4321 + n))
        (_, ci), ms_ref = _event_ms(torch, dev, lambda: orc.forward(w, x), reps=1)
        (_, ck), ms_ours = _event_ms(torch, dev, lambda: model(x), reps=3)
        res[str(n)] = {"stock_pytorch_tokens_per_s": n / ms_ref * 1e3, "stock_pytorch_ms": ms_ref,
                       "rqae_b200_tokens_per_s": n / ms_ours * 1e3, "rqae_b200_ms": ms_ours,
                       "speedup": ms_ref / ms_ours,
                       "tokens_with_identical_codes": float((ci == ck).all(-1).float().mean().item())}
        del x, ci, ck
    res["note"] = ("stock PyTorch = oracle/rqae_oracle.forward (the reference's ATen calls, op for op) on cuda tensors, "
                   "torch %s; both on the same B200, CUDA events; code disagreements are near-tie flips of a different "
                   "fp32 summation order (cuBLAS vs the fused kernel), see `parity`" % torch.__version__)
    return res


def config3_9b_extra(torch, dist, dev, rank, world, tokens):
    """BASELINE configs[3]: Gemma-2-9B width (d=3584), deeper stack (nq=2048), encode-only code extraction;
    every rank encodes its own `tokens` tokens (weak scaling), time = max over ranks."""
    from rqae_b200 import RQAE
    torch.manual_seed(0)
    m = RQAE(dim=3584, num_quantizers=2048).eval().to(dev)
    m.freeze_packed()
    x = torch.empty(1, tokens, 3584, device=dev)
    gen = torch.Generator(device=dev).manual_seed(99 + rank)
    for c0 in range(0, tokens, 1 << 16):
        c1 = min(tokens, c0 + (1 << 16))
        x[0, c0:c1] = torch.randn(c1 - c0, 3584, generator=gen, device=dev)
    m.encode(x[:, : min(tokens, 1 << 15)], out_dtype=torch.int16)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    codes = m.encode(x, out_dtype=torch.int16)
    b.record()
    torch.cuda.synchronize(dev)
    ms = a.elapsed_time(b)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    flop_tok = 2048 * (2 * 2 * 4 * 3584 + 5000 + 3584)
    res = {"tokens_per_gpu": tokens, "n_gpus": world, "dim": 3584, "num_quantizers": 2048, "code_dtype": "int16",
           "tokens_per_s": world * tokens / ms * 1e3, "tokens_per_s_per_gpu": tokens / ms * 1e3, "ms": ms,
           "tflops_fp32_per_gpu": flop_tok * tokens / ms / 1e9, "flop_per_token": flop_tok,
           "checksum_codes": int(codes[0, :4096].long().sum().item())}
    del m, x, codes
    torch.cuda.empty_cache()
    return res


def config3_9b_cpu_port(torch, tokens=32):
    from oracle import rqae_oracle as orc
    w = orc.random_init(dim=3584, num_quantizers=2048)
    x = torch.randn(1, tokens, 3584, generator=torch.Generator().manual_seed(3))
    orc.forward(w, x[:, :4])
    t0 = time.perf_counter()
    orc.forward(w, x)
    dt = time.perf_counter() - t0
    return {"tokens_per_s": tokens / dt, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{tokens} tokens, full depth (nq=2048), forward incl. reconstruction, torch CPU fp32, {dt:.1f} s"}


def config4_mining_extra(torch, dist, model, x, dev, rank, world, tokens, n_features=1024, group=256, top_k=100):
    """BASELINE configs[4] (scripts/3_make_rqae_features.py pattern) at its stated scale: every rank encodes its
    `tokens` tokens (2 Mi per GPU = 16 Mi on 8 GPUs), then for feature groups of `group`: intensities of the group over
    the rank's tokens at the 14 cuts of scripts/3:178 (tcgen05 GEMM), all_to_all so that every (feature, cut) row is
    whole on one rank (shard.exchange_to_feature_shards), top / middle / bottom-100 of every row over ALL tokens
    (radix select).  Wall clock from a barrier to the last kernel, max over ranks; stage times are CUDA events."""
    from rqae_b200.feature import intensity_many, select_top_middle_bottom, layer_weights_f16, IntensityWorkspace
    from rqae_b200 import shard
    iws = IntensityWorkspace()     # feature groups run over the same codes: their tile-major copy is made once
    T_x = x.shape[1]
    ev = lambda: torch.cuda.Event(enable_timing=True)
    codes = torch.empty(tokens, NQ, dtype=torch.int16, device=dev)
    lw = layer_weights_f16(model).to(dev)
    buf = torch.empty(group, len(SCRIPT3_CUTS), (tokens + 255) // 256 * 256, dtype=torch.float16, device=dev)
    # One untimed pass of a feature group over whatever the buffers hold (the warm-up of this extra): NCCL brings up its
    # point-to-point channels lazily and per message size, and the caching allocator has to obtain the 15 GB receive and
    # repack buffers once; both cost 100-200 ms on first use and belong to a cold process, not to the path.
    codes.zero_()
    wu = intensity_many(model, codes, codes[:group].to(torch.int32), SCRIPT3_CUTS, layer_weights=lw, out=buf)
    if world > 1:
        wu, _ = shard.exchange_to_feature_shards(wu, world * tokens)
    select_top_middle_bottom(wu, top_k)
    del wu
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t_wall0 = time.perf_counter()
    e0, e1 = ev(), ev()
    e0.record()
    gen = torch.Generator(device=dev).manual_seed(777 + rank)
    for c0 in range(0, tokens, T_x):
        n = min(T_x, tokens - c0)
        if c0 > 0:   # fresh activations for every pass over the staging buffer
            for k0 in range(0, n, 1 << 16):
                k1 = min(n, k0 + (1 << 16))
                x[0, k0:k1] = torch.randn(k1 - k0, D, generator=gen, device=dev)
        codes[c0:c0 + n] = model.encode(x[:, :n], out_dtype=torch.int16)[0]
    e1.record()
    # feature centers = the codes of n_features tokens (of rank 0's shard), the same on every rank
    pick = torch.randperm(tokens, generator=torch.Generator().manual_seed(5))[:n_features].to(dev)
    centers = codes[pick].to(torch.int32)
    if world > 1:
        dist.broadcast(centers, src=0)
    n_total = world * tokens
    ms_int = ms_x = ms_sel = 0.0
    ms_x_groups = []
    checksum = 0
    ms_int_groups = []
    for f0 in range(0, n_features, group):
        a, b, c, d = ev(), ev(), ev(), ev()
        a.record()
        inten = intensity_many(model, codes, centers[f0:f0 + group], SCRIPT3_CUTS, layer_weights=lw, out=buf, workspace=iws)
        b.record()
        if world > 1:
            rows, _ = shard.exchange_to_feature_shards(inten, n_total)
        else:
            rows = inten
        c.record()
        idx, val = select_top_middle_bottom(rows, top_k)
        d.record()
        torch.cuda.synchronize(dev)
        ms_int += a.elapsed_time(b); ms_x += b.elapsed_time(c); ms_sel += c.elapsed_time(d)
        ms_x_groups.append(round(b.elapsed_time(c), 2))
        ms_int_groups.append(round(a.elapsed_time(b), 2))
        checksum += int(idx[:, :, 0, 0].sum().item())
        del rows, idx, val
    t_wall = time.perf_counter() - t_wall0
    ms_enc = e0.elapsed_time(e1)
    stats = torch.tensor([t_wall, ms_enc, ms_int, ms_x, ms_sel], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    t_wall, ms_enc, ms_int, ms_x, ms_sel = [float(v) for v in stats.tolist()]
    rows_per_rank = (n_features // world) * len(SCRIPT3_CUTS)
    peaks = measured_peaks()
    res = {"tokens_per_gpu": tokens, "tokens_total": n_total, "n_gpus": world, "features": n_features, "cuts": len(SCRIPT3_CUTS),
           "top_k": top_k, "feature_group": group,
           "tokens_per_s": n_total / t_wall, "seconds": t_wall,
           "stage_ms_max_over_ranks": {"encode": ms_enc, "intensity_gemm": ms_int, "all_to_all_and_repack": ms_x, "select": ms_sel},
           "encode_tokens_per_s": n_total / ms_enc * 1e3,
           "intensity_tflops_per_gpu": 2.0 * tokens * n_features * 4 * (SCRIPT3_CUTS[-1] + 1) / ms_int / 1e9,
           "intensity_frac_of_tensor_peak": 2.0 * tokens * n_features * 4 * (SCRIPT3_CUTS[-1] + 1) / ms_int / 1e9
                                            / (peaks["bf16_tflops"] if peaks else 1590.0),
           "select_gbs_per_gpu": rows_per_rank * n_total * 2 / ms_sel / 1e6,
           "exchange_gbs_per_gpu": (n_features * len(SCRIPT3_CUTS) * tokens * 2 * (world - 1) / world) / ms_x / 1e6 if world > 1 else None,
           "exchange_ms_per_group_rank0": ms_x_groups, "intensity_ms_per_group_rank0": ms_int_groups, "checksum_top_idx": checksum,
           "timing": "host wall clock barrier -> last kernel done (encode + feature groups x (GEMM, all_to_all, select)), "
                     "max over ranks"}
    del codes, buf
    torch.cuda.empty_cache()
    return res


def dump_outputs(torch, out_dir, q, codes):
    """quantized_out (1, T, D) and indices (1, T, nq) of RQAE.forward at DUMP_ROWS token rows (all of them when
    T is smaller), ascending; the rows are drawn from a fixed seed and depend on T alone."""
    import numpy as np
    rows = torch.randperm(codes.shape[1], generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    rows = rows.to(codes.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "quantized_out.npy"), q[0, rows].cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "indices.npy"), codes[0, rows].cpu().numpy().astype(np.float64))


def run_b200(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from rqae_b200 import RQAE, _lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL announces itself on stdout when NCCL_DEBUG is set in the environment; stdout carries exactly one
        # JSON line, so route fd 1 to stderr while the communicator comes up
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    lib = _lib.load()

    torch.manual_seed(0)
    model = RQAE().eval().to(dev)       # same parameters as torch.manual_seed(0); reference RQAE()
    model.freeze_packed()
    T = args.tokens
    gen = torch.Generator(device=dev).manual_seed(1234 + rank * 1000)
    x = torch.empty(T, D, device=dev)
    for c0 in range(0, T, 1 << 16):
        c1 = min(T, c0 + (1 << 16))
        x[c0:c1] = torch.randn(c1 - c0, D, generator=gen, device=dev)
    xv = x.view(1, T, D)

    def barrier():
        if world > 1:
            dist.barrier()

    # ---- parity gate: the reference's 4096-token KAT through this very model object ----
    par = None
    if rank == 0 and not args.no_parity:
        par = parity_block(torch, model, dev)

    for _ in range(max(args.warmup, 3)):
        q, codes = model(xv)
    torch.cuda.synchronize(dev)
    del q, codes

    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    torch.cuda.synchronize(dev)
    lib.rqae_launch_count(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        q, codes = model(xv)
    e1.record()
    torch.cuda.synchronize(dev)
    barrier()
    launches = int(lib.rqae_launch_count(0))
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    checksum = int(codes.sum().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, args.dump_outputs, q, codes)
    del q, codes
    ms_step = ms / args.steps
    value = world * T / (ms_step * 1e-3)

    # ---- end to end through the host-buffer API ----
    e2e = None
    if not args.no_e2e:
        import psutil
        Te = args.e2e_tokens or T
        need = Te * (4 * D * 2 + 8 * NQ + 4 * NQ)
        avail = psutil.virtual_memory().available / max(1, world)
        while need > 0.25 * avail and Te > (1 << 16):
            Te //= 2
            need = Te * (4 * D * 2 + 8 * NQ + 4 * NQ)
        xh = torch.empty(Te, D, dtype=torch.float32, pin_memory=True)
        for c0 in range(0, Te, 1 << 16):
            c1 = min(Te, c0 + (1 << 16))
            xh[c0:c1].copy_(x[c0 % T:c0 % T + (c1 - c0)] if c0 % T + (c1 - c0) <= T else torch.randn(c1 - c0, D))
        # result buffers are allocated (page-locked) once, as a caller that loops over shards would
        qh = torch.empty(Te, D, dtype=torch.float32, pin_memory=True)
        steps_e = args.e2e_steps or min(args.steps, 3)

        def e2e_run(dt, want_q=True):
            ch = torch.empty(Te, NQ, dtype=dt, pin_memory=True)
            model.forward_host(xh[: 1 << 15], out=(qh[: 1 << 15], ch[: 1 << 15]), out_dtype=dt, want_q=want_q)  # warm-up of the host path
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps_e):
                model.forward_host(xh, out=(qh, ch), out_dtype=dt, want_q=want_q)
            t_e = time.perf_counter() - t0    # forward_host returns after the last D2H copy completed
            barrier()
            if world > 1:
                t = torch.tensor([t_e], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                t_e = float(t.item())
            return world * Te * steps_e / t_e, int(ch[: 1 << 12].long().sum().item())

        import ctypes
        v64, ck64 = e2e_run(torch.int64)
        v32, ck32 = e2e_run(torch.int32)
        venc, ckenc = e2e_run(torch.int32, want_q=False)
        m_, t_ = ctypes.c_int(0), ctypes.c_int(0)
        lib.rqae_forward_host_mode(ctypes.byref(m_), ctypes.byref(t_))
        narrow = m_.value == 1
        e2e = {"value": v64, "unit": UNIT, "h2d_bytes_per_step": Te * D * 4,
               "d2h_bytes_per_step": Te * ((NQ * 2 if narrow else NQ * 8) + D * 4), "tokens_per_step_per_gpu": Te,
               "steps": steps_e, "result_bytes_per_step": Te * (NQ * 8 + D * 4),
               "code_transfer": "narrow" if narrow else "direct", "widen_threads": t_.value if narrow else 0,
               "timing": "host wall clock around RQAE.forward_host (pinned host buffers in and out; H2D, kernel and "
                         "D2H of 9472-token chunks on three streams inside the C library; "
                         + ("codes cross PCIe as int16 and are widened into the caller's int64 tensor by %d host "
                            "thread(s) while the next chunk is in flight; " % t_.value if narrow else
                            "int64 codes written by the kernel and copied straight into the caller's tensor; ")
                         + "returns after the last D2H), max over ranks",
               "checksum_codes": ck64,
               "int32_codes": {"value": v32, "unit": UNIT, "d2h_bytes_per_step": Te * ((NQ * 2 if narrow else NQ * 4) + D * 4),
                               "checksum_codes": ck32,
                               "note": "same call with out_dtype=int32, the dtype the reference's code store keeps "
                                       "(scripts/1_create_activations.py:184-186)"},
               "encode_only_int32_codes": {"value": venc, "unit": UNIT, "d2h_bytes_per_step": Te * NQ * (2 if narrow else 4),
                                           "checksum_codes": ckenc,
                                           "note": "code extraction only (forward_host(want_q=False)): what scripts/1 keeps of the "
                                                   "RQAE output; no reconstruction crosses PCIe, so the host link carries 9.2 KB in "
                                                   "and 2 KB out per token -- the variant that shows the pipeline itself scales "
                                                   "when the device->host bytes do not bind (DESIGN.md 7)"}}
        del xh, qh

    # ---- side measurements (outside the timed region) ----
    extra = None
    if rank == 0:
        Ts = min(T, 1 << 18)
        xs = xv[:, :Ts]
        def timed(fn, reps=2):
            fn(); torch.cuda.synchronize(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                out = fn()
            b.record(); torch.cuda.synchronize(dev)
            return out, Ts * reps / (a.elapsed_time(b) * 1e-3)
        codes_s, enc_rate = timed(lambda: model.encode(xs, out_dtype=torch.int16))
        dec_exact, dec_rate = timed(lambda: model.decode(codes_s))
        extra = {"encode_only_int16_tokens_per_s": enc_rate, "decode_only_tokens_per_s": dec_rate, "tokens": Ts,
                 "decode_frac_of_fp32_peak": None}
        if not args.no_extras and world == 1:
            try:   # opt-in tensor-core decode (tcgen05 GEMM over the codes), not bit-exact: rate and error vs the exact kernel
                tc = {}
                for prec, npass in (("f16", 1), ("f16x3", 3)):
                    dq, rate = timed(lambda: model.decode(codes_s, precision=prec))
                    tc[prec] = {"tokens_per_s": rate, "algorithmic_tflops": rate * 2 * 4 * NQ * D / 1e12,
                                "issued_tflops": rate * npass * 2 * 4 * NQ * D / 1e12, "passes": npass,
                                "max_err_over_max_abs": float(((dq - dec_exact).abs().max() / dec_exact.abs().max()).item())}
                    del dq
                extra["decode_tensor_core_opt_in"] = tc
            except Exception as e:
                extra["decode_tensor_core_opt_in"] = {"error": repr(e)}
        del dec_exact
        if not args.no_extras and world == 1:
            for name, fn in (("mining", lambda: mining_extras(torch, model, codes_s[0, : 1 << 17], dev)),
                             ("hook_512", lambda: hook_extra(torch, model, dev)),
                             ("stock_pytorch_gpu", lambda: stock_pytorch_gpu_extra(torch, model, dev)),
                             ("example_search", lambda: search_extras(torch, model, dev))):
                try:
                    extra[name] = fn()
                except Exception as e:   # side measurement only: never lose the bench line over it
                    extra[name] = {"error": repr(e)}
                torch.cuda.empty_cache()
        del codes_s
    # configs[3] and configs[4] run on EVERY rank (weak scaling, max over ranks)
    if not args.no_extras:
        try:
            c4 = config4_mining_extra(torch, dist, model, xv, dev, rank, world, args.tokens_mining)
        except Exception as e:
            c4 = {"error": repr(e)}
        del x, xv
        torch.cuda.empty_cache()
        try:
            c3 = config3_9b_extra(torch, dist, dev, rank, world, args.tokens_9b)
        except Exception as e:
            c3 = {"error": repr(e)}
        if rank == 0:
            extra["config3_9b"] = c3
            extra["config4_mining"] = c4
            if world == 1:
                try:
                    extra["config3_9b"]["cpu_port"] = config3_9b_cpu_port(torch)
                except Exception as e:
                    extra["config3_9b"]["cpu_port"] = {"error": repr(e)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    fp32 = fp32_peak_tflops(torch, lib, dev)
    fp32_peak = max(fp32["ffma2"], fp32["ffma"])
    ach_tflops = FLOP_PER_TOKEN_FWD * T / (ms_step * 1e-3) / 1e12
    ach_gbs = HBM_BYTES_PER_TOKEN_FWD * T / (ms_step * 1e-3) / 1e9
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "forward_traffic.json")))
        if int(tj.get("tokens_per_launch", 0)) == T:
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
    except Exception:
        pass
    if extra is not None:
        # algorithmic flops of decode (SURVEY 8d): 2*4*D + D = 20 736 per layer-token; the kernel issues 12*D
        extra["decode_frac_of_fp32_peak"] = extra["decode_only_tokens_per_s"] * NQ * (2 * 4 * D + D) / 1e12 / fp32_peak
        extra["decode_fp32_pipe_busy_frac"] = extra["decode_only_tokens_per_s"] * NQ * (6 * D) * 2 / 1e12 / fp32_peak
        tcx = extra.get("decode_tensor_core_opt_in")
        if isinstance(tcx, dict) and peaks:
            for v in tcx.values():
                if isinstance(v, dict) and "algorithmic_tflops" in v:
                    v["algorithmic_frac_of_tensor_peak"] = v["algorithmic_tflops"] / peaks["bf16_tflops"]
        c3 = extra.get("config3_9b")
        if isinstance(c3, dict) and "tflops_fp32_per_gpu" in c3:
            c3["frac_of_fp32_peak"] = c3["tflops_fp32_per_gpu"] / fp32_peak
    roofline = {
        "kernel": "rq::rq_forward_kernel (E=9 instantiation for d=2304; one cooperative launch per step)",
        "bound": "fp32", "achieved": ach_tflops, "peak": fp32_peak, "unit": "TFLOP/s", "frac": ach_tflops / fp32_peak,
        "peak_source": "measured live: rqae_fp32_peak_probe, best of FFMA2 %.1f / FFMA %.1f TFLOP/s" % (fp32["ffma2"], fp32["ffma"]),
        "operand_pattern_ceiling": {"inproj_sweep": fp32["pattern_inproj"], "outproj_sweep": fp32["pattern_outproj"],
                                    "unit": "TFLOP/s",
                                    "note": "what the FMA pipe delivers for the kernel's own FFMA2 operand mix (scalar weight "
                                            "x token pair + pair) with all operands in registers: the register-file "
                                            "read ports cap it below the dense peak; the fraction above is still quoted "
                                            "against the dense peak"},
        "flop_per_token": FLOP_PER_TOKEN_FWD, "traffic": traffic,
        "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of one launch of this size (ncu, "
                        "profiles/forward_traffic.json); algorithmic bytes per launch = %d" % (HBM_BYTES_PER_TOKEN_FWD * T),
        "why_not_hbm_or_tensor": "bit-exact fp32 parity confines the layer recurrence to the FP32 FMA pipe "
                                 "(arithmetic intensity 1787 FLOP/B; TF32/bf16 splits flip codes, see DESIGN.md)",
        "hbm": {"achieved": ach_gbs, "peak": peaks["hbm_gbs"] if peaks else 6650.0, "unit": "GB/s",
                "frac": ach_gbs / (peaks["hbm_gbs"] if peaks else 6650.0),
                "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)",
                "bytes_per_token": HBM_BYTES_PER_TOKEN_FWD},
        "tensor": {"achieved": ach_tflops, "peak": peaks["bf16_tflops_sustained"] if peaks else 1400.0,
                   "unit": "TFLOP/s", "frac": ach_tflops / (peaks["bf16_tflops_sustained"] if peaks else 1400.0),
                   "peak_source": "MEASURED_PEAKS.json (sustained)" if peaks else "fallback"},
    }
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "BASELINE configs[1]: random-init RQAE (torch.manual_seed(0)) d=2304 cd=4 K=625 nq=1024, "
                               "forward = encode (int64 codes) + fp32 reconstruction of synthetic N(0,1) tokens",
                   "tokens_per_gpu_per_step": T, "dim": D, "num_quantizers": NQ,
                   "parallelism": f"token-sharded dp{world}, no collective on the data path",
                   "l2": "per-step inputs+outputs (%.1f GB) exceed the 126 MB L2; the 85 MB of weights are L2-resident by design"
                         % (HBM_BYTES_PER_TOKEN_FWD * T / 1e9)},
        "roofline": roofline, "clocks": clocks, "gpu_launches": launches, "e2e": e2e, "checksum_codes": checksum,
        "parity": par, "extra": extra,
    }
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(args.cpu_seconds)
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if par is not None and (par.get("failures", 0) > 0 or "error" in par):
        raise SystemExit("parity gate failed: %s" % json.dumps(par)[:400])


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
