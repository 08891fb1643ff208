"""One-process GPU check of the nearest-example search (SURVEY 8f-3): the parity tests of tests/test_search_gpu.py,
then stage timings at the reference's dataset shape (36 864 sequences x 127 positions x 1024 layers, server.py:139),
written line by line to gpurun_out/search_check.jsonl so that a call cut short still leaves what it measured.

    gpurun --timeout 240 -- 'python tools/gpu_search.py'
"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "gpurun_out", "search_check.jsonl")
os.makedirs(os.path.dirname(OUT), exist_ok=True)


def emit(**kw):
    with open(OUT, "a") as f:
        f.write(json.dumps(kw) + "\n")
    print(json.dumps(kw), flush=True)


def timed(fn, st):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    r = fn()
    e1.record(st)
    e1.synchronize()
    return r, e0.elapsed_time(e1)


def bench(N, S=127, nq=1024, K=625, Sq=127, reps=2):
    import torch
    from rqae_b200 import _lib
    from rqae_b200.feature import select_top_middle_bottom
    from rqae_b200.search import IntensityEngine, SERVER_LAYERS
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(1)
    sims = (torch.randn(nq, K, K, generator=g, device=dev, dtype=torch.float16) * 0.25)
    sims.diagonal(dim1=1, dim2=2).fill_(1.0)          # a code matches itself best, as a cosine table does
    codes = torch.randint(0, K, (N, S, nq), generator=g, device=dev, dtype=torch.int16)
    eng = IntensityEngine(sims=sims, activations=codes)
    idx = N // 3
    layers = SERVER_LAYERS
    q = eng._query(idx, None, max(layers))
    lib = _lib.load()
    st = torch.cuda.current_stream(dev)
    best = None
    for rep in range(reps + 1):
        torch.cuda.synchronize()
        lib.rqae_launch_count(1)
        t_sel = 0.0
        it = eng.accumulate(q, layers)
        stages = []
        t_all0 = time.perf_counter()
        e_begin, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e_begin.record(st)
        prev = torch.cuda.Event(enable_timing=True)
        prev.record(st)
        for layer, (acc, maxv) in zip(layers, it):
            mid = torch.cuda.Event(enable_timing=True)
            mid.record(st)
            sel, _ = select_top_middle_bottom(maxv, 30)
            end = torch.cuda.Event(enable_timing=True)
            end.record(st)
            stages.append((layer, prev, mid, end))
            prev = end
        e_end.record(st)
        e_end.synchronize()
        total = e_begin.elapsed_time(e_end)
        per = [{"layer": l, "accumulate_max_ms": round(a.elapsed_time(b), 3), "select_ms": round(b.elapsed_time(c), 3)}
               for l, a, b, c in stages]
        launches = int(lib.rqae_launch_count(0))
        if rep > 0 and (best is None or total < best["total_ms"]):
            best = {"total_ms": total, "stages": per, "launches": launches, "wall_ms": (time.perf_counter() - t_all0) * 1e3}
    # property at full size: the query sequence is the top example of each of its own positions at the last layer
    self_top = bool((sel[:, 0, 0] == idx).all().item())
    rows = N * S * max(layers)
    emit(what="search_bench", sequences=N, positions=S, layers=max(layers), query_positions=Sq, K=K,
         total_ms=round(best["total_ms"], 3), wall_ms=round(best["wall_ms"], 3), launches=best["launches"],
         sequences_per_s=round(N / (best["total_ms"] * 1e-3), 1),
         table_row_TBps=round(rows * 256 / (best["total_ms"] * 1e-3) / 1e12, 3),
         code_store_GBps=round(rows * 2 / (best["total_ms"] * 1e-3) / 1e9, 2),
         self_match_top1=self_top, stages=best["stages"])
    del eng, codes, sims
    torch.cuda.empty_cache()


def main():
    t0 = time.time()
    if "--no-tests" not in sys.argv:
        import pytest
        rc = pytest.main(["-x", "-q", "-m", "gpu", os.path.join(ROOT, "tests", "test_search_gpu.py"), "-p", "no:cacheprovider"])
        emit(what="pytest tests/test_search_gpu.py", exit_code=int(rc), seconds=round(time.time() - t0, 1))
        if int(rc) != 0:
            return int(rc)
    if "--bench-extra" in sys.argv:        # the exact function bench.py runs as extra["example_search"], on the 2B model
        import torch
        import bench
        from rqae_b200 import RQAE
        dev = torch.device("cuda:0")
        torch.manual_seed(0)
        model = RQAE().eval().to(dev)
        try:
            emit(what="bench.search_extras", **bench.search_extras(torch, model, dev))
        except Exception as e:
            emit(what="bench.search_extras", error=repr(e))
            return 1
        return 0
    sizes = [int(a) for a in sys.argv[1:] if a.isdigit()] or [2048, 36864]
    for N in sizes:
        try:
            bench(N)
        except Exception as e:   # recorded, not hidden
            emit(what="search_bench", sequences=N, error=repr(e))
            return 1
    return 0


if __name__ == "__main__":
    sys.exit(main())
