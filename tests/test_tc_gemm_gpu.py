"""The tcgen05 GEMM kernel ``rq_intensity_kernel`` (rq_intensity.cuh) against exact emulations of its own arithmetic, at
shapes where every CTA runs several units: feature intensities (EPI 0, ``intensity_many``), the tensor-core decode (EPI 1,
``RQAE.decode(precision="f16" / "f16x3")``) and the tensor-core search maxima (EPI 2, ``IntensityEngine(precision="tc")``).

Every operand of these kernels is an fp16 value that can be computed on the host, and every product of two fp16 values is
exact; the only freedom is the order of the tensor core's fp32 accumulation.  The emulators below reproduce the kernels'
operand roundings (not the reference's) in float64 torch on any device.  ``acc`` is the exact sum and ``S`` the sum of the
absolute products; every map from the accumulator to the output (fp16 rounding, multiply by a positive reciprocal, fp32
add, max) is monotone, so each test asserts the bracket

    emul(acc - B) <= kernel <= emul(acc + B),   B = 4 * nkb * 2^-23 * S

element by element, nkb = the K-blocks (64 k values, four 16-deep MMAs) up to the cut: two fp32 ulps of S per MMA.  Each
test prints the worst |kernel - emul(acc)| in units of the bracket's half-width on that side (emul(acc +- B) - emul(acc)
in the output's own type), the fraction of elements where the bracket holds more than one output value, and the fraction
bit-equal to emul(acc).

Measured on a B200 (148 SMs, 1000 W power limit): the bracket held for every value checked, and no kernel value left
emul(acc) by more than the bracket's width (worst ratio 1.000).  Bit-equal to emul(acc): 0.9978 of the production
intensity shape (bracket wider than one value for 0.34 of them), 0.9993 with 64 cuts, 0.962 at NKB = 200 (where B spans
several fp16 steps for every value), >= 0.998 for the other intensity shapes and 0.9988-0.9998 for the search maxima.
The decode's fp32 output is finer than B: there the kernel stayed within 0.02-0.033 of B of emul(acc) (0.1-0.8 % of
the values bit-equal), so B is an upper bound, not a measurement, of the tensor core's accumulation error.
"""
import math
import os
import time

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import feature_oracle as fo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ATOL = 2e-3                      # the reference-form tolerance of tests/test_feature_gpu.py
EPS32 = 2.0 ** -23
TOK = 256                        # tokens per unit of the intensity / decode kernels
SCRIPT3_LAYERS = [2, 4, 6, 8, 12, 16, 24, 32, 48, 64, 128, 256, 512, 1023]


# ---------------------------------------------------------------------------------------------------------------------
# emulators
# ---------------------------------------------------------------------------------------------------------------------
def _clamp_codes(c: torch.Tensor, K: int, wrap_negative: bool = False) -> torch.Tensor:
    """The kernels map every code outside [0, K) (negative, >= K, any int64) to row K, the zero row; the decode first
    turns a code in [-K, 0) into the python-style index c + K, as codebook[0][codes] does."""
    c = c.long()
    if wrap_negative:
        c = torch.where(c < 0, c + K, c)
    return torch.where((c >= 0) & (c < K), c, torch.full_like(c, K))


def weight_prefixes(w16: torch.Tensor, cuts):
    """int_prep_kernel: wc_c = fp16(sequential fp32 sum of the fp16 weights up to cut_c), inv_c = fp32(1 / wc_c)."""
    w = w16.detach().cpu().to(torch.float16).numpy()
    run, l, wc, inv = np.float32(0), 0, [], []
    for c in cuts:
        while l <= c:
            run = np.float32(run + np.float32(w[l]))
            l += 1
        h = np.float32(np.float16(run))
        wc.append(h)
        inv.append(np.float32(1) / h)
    return np.array(wc, np.float32), np.array(inv, np.float32)


class IntensityEmu:
    """int_prep_kernel / int_pack_u_kernel / finish2 / finish_packed for sorted unique ``cuts``.

    U[f][l][j] = fp16(fp32(w_l * n[center_f,l][j])), V[t][l][j] = fp16(n[code_t,l][j]), zero outside [0, K);
    acc[f][c][t] = sum over l <= cut_c and j of U V (float64: exact products, negligible sum error);
    out = fp16(fp32(fp16(acc)) * inv_c)."""

    def __init__(self, cb0: torch.Tensor, w16: torch.Tensor, cuts, dev):
        self.cuts = sorted(set(int(c) for c in cuts))
        self.L = L = self.cuts[-1] + 1
        n = F.normalize(cb0.detach().to(device=dev, dtype=torch.float32), dim=-1)   # intensity_many's own call
        self.K = K = n.shape[0]
        wl = w16[:L].to(device=dev, dtype=torch.float16).float()
        z = torch.zeros(L, 1, 4, dtype=torch.float64, device=dev)
        self.ut = torch.cat([(wl[:, None, None] * n[None]).half().double(), z], 1)     # (L, K + 1, 4)
        self.vt = torch.cat([n.half().double(), z[0]], 0)                               # (K + 1, 4)
        self.segs, self.nkb, prev, kb = [], [], -1, 0
        for c in self.cuts:
            self.segs.append((prev + 1, c + 1))
            kb += (c - prev + 15) // 16
            self.nkb.append(kb)
            prev = c
        self.wc, inv = weight_prefixes(w16, self.cuts)
        self.inv = torch.from_numpy(inv).to(dev)
        self.dev = dev

    def acc(self, centers: torch.Tensor, codes: torch.Tensor, with_s: bool = True):
        """centers (F, >= L), codes (T, >= L) integer -> acc, S (F, C, T) float64."""
        L = self.L
        c = _clamp_codes(centers[:, :L].to(self.dev), self.K)
        t = _clamp_codes(codes[:, :L].to(self.dev), self.K)
        U = self.ut[torch.arange(L, device=self.dev)[None], c]       # (F, L, 4)
        V = self.vt[t]                                                # (T, L, 4)
        ra = torch.zeros(U.shape[0], V.shape[0], dtype=torch.float64, device=self.dev)
        rs = torch.zeros_like(ra) if with_s else None
        accs, ss = [], []
        for a, b in self.segs:
            u, v = U[:, a:b].reshape(U.shape[0], -1), V[:, a:b].reshape(V.shape[0], -1)
            ra = ra + u @ v.T
            accs.append(ra)
            if with_s:
                rs = rs + u.abs() @ v.abs().T
                ss.append(rs)
        return torch.stack(accs, 1), (torch.stack(ss, 1) if with_s else None)

    def out(self, x: torch.Tensor) -> torch.Tensor:
        return (x.float().half().float() * self.inv[None, :, None]).half()

    def bracket(self, acc, S):
        B = 4 * torch.tensor(self.nkb, dtype=torch.float64, device=self.dev)[None, :, None] * EPS32 * S
        return self.out(acc - B), self.out(acc), self.out(acc + B)


def _h_rem(v: torch.Tensor) -> torch.Tensor:
    """dec_prep_kernel / dec_pack_u_kernel: fp16(v - fp16(v)), the difference taken in fp32."""
    v = v.float()
    return (v - v.half().float()).half()


class DecodeEmu:
    """dec_prep_kernel / dec_pack_u_kernel / dec_bias_kernel: V = codebook0[code] and U = W_out as fp16 (passes = 1), plus
    V_hi U_lo + V_lo U_hi (passes = 3); bias_d = sequential fp32 sum of b_out[l][d] over the selected layers;
    out = fp32(fp32(acc) + bias_d)."""

    def __init__(self, model, passes: int, layers, nq_codes: int, dev):
        self.passes, self.L, self.dev = passes, nq_codes, dev
        cb0 = model.codebook.detach()[0].to(device=dev, dtype=torch.float32)
        self.K = K = cb0.shape[0]
        z = torch.zeros(1, 4, dtype=torch.float64, device=dev)
        self.vhi = torch.cat([cb0.half().double(), z])
        self.vlo = torch.cat([_h_rem(cb0).double(), z])
        w = torch.stack([l[1].weight.detach() for l in model.layers])[:nq_codes].to(device=dev, dtype=torch.float32)
        b = torch.stack([l[1].bias.detach() for l in model.layers])[:nq_codes].to(device=dev, dtype=torch.float32)
        sel = [l for l in range(nq_codes) if layers is None or l in layers]
        mask = torch.zeros(nq_codes, dtype=torch.float64, device=dev)
        mask[sel] = 1
        D = w.shape[1]
        self.uhi = (w.half().double() * mask[:, None, None]).permute(1, 0, 2).reshape(D, -1)     # (D, 4 L)
        self.ulo = (_h_rem(w).double() * mask[:, None, None]).permute(1, 0, 2).reshape(D, -1)
        bias = torch.zeros(D, dtype=torch.float32, device=dev)
        for l in sel:
            bias = bias + b[l]
        self.bias = bias
        self.nkb = passes * ((nq_codes + 15) // 16)

    def acc(self, codes: torch.Tensor):
        t = _clamp_codes(codes[:, :self.L].to(self.dev), self.K, wrap_negative=True)
        vh = self.vhi[t].reshape(t.shape[0], -1)
        acc, S = vh @ self.uhi.T, vh.abs() @ self.uhi.abs().T
        if self.passes == 3:
            vl = self.vlo[t].reshape(t.shape[0], -1)
            acc = acc + vh @ self.ulo.T + vl @ self.uhi.T
            S = S + vh.abs() @ self.ulo.abs().T + vl.abs() @ self.uhi.abs().T
        return acc, S                                                            # (T, D)

    def out(self, x: torch.Tensor) -> torch.Tensor:
        return x.float() + self.bias

    def bracket(self, acc, S):
        B = 4 * self.nkb * EPS32 * S
        return self.out(acc - B), self.out(acc), self.out(acc + B)


def search_emu(eng, query: torch.Tensor, layers, seqs: slice):
    """rq_intensity_kernel<2> with srch_prep_kernel / srch_pack_u_kernel: prefix[c][q][t] = sum over l < layers[c] and j of
    utab[l][query_q,l][j] * vtab[l][code_t,l][j] from the engine's own fp16 tables; out = fp16(max over the positions of a
    sequence).  Returns lo, mid, hi (C, Sq, n) fp16 and the float64 maxima of the exact prefix."""
    dev = eng.sims.device
    K = eng.sims.shape[1]
    last = layers[-1]
    ut, vt = eng._utab.double(), eng._vtab.double()
    ar = torch.arange(last, device=dev)
    Uq = ut[ar[None], _clamp_codes(query[:, :last].to(dev), K)]                 # (Sq, last, 8)
    codes = eng.activations[seqs]
    n, S = codes.shape[:2]
    V = vt[ar[None], _clamp_codes(codes.reshape(n * S, -1)[:, :last], K)]       # (n S, last, 8)
    ra = torch.zeros(n * S, Uq.shape[0], dtype=torch.float64, device=dev)
    rs = torch.zeros_like(ra)
    lo, mid, hi, mx = [], [], [], []
    a, kb = 0, 0
    for b in layers:
        u, v = Uq[:, a:b].reshape(Uq.shape[0], -1), V[:, a:b].reshape(n * S, -1)
        ra = ra + v @ u.T
        rs = rs + v.abs() @ u.abs().T
        kb += (b - 1) // 8 - a // 8 + 1
        B = 4 * kb * EPS32 * rs
        for dst, x in ((lo, ra - B), (mid, ra), (hi, ra + B)):
            dst.append(x.view(n, S, -1).max(dim=1).values.T.float().half())
        mx.append(ra.view(n, S, -1).max(dim=1).values.T)
        a = b
    return torch.stack(lo), torch.stack(mid), torch.stack(hi), torch.stack(mx)


class Bracket:
    """Collects the check over several chunks; ``report`` prints the three numbers and asserts."""

    def __init__(self, name):
        self.name, self.n, self.bad, self.ties, self.equal, self.worst, self.first_bad = name, 0, 0, 0, 0, 0.0, None

    def add(self, got, lo, mid, hi, where=""):
        g, l, m, h = (t.double() for t in (got, lo, mid, hi))
        ok = (l <= g) & (g <= h)
        d = (g - m).abs()
        w = torch.where(g >= m, h - m, m - l)
        ratio = torch.where(d == 0, torch.zeros_like(d), d / w)
        self.n += g.numel()
        nb = int((~ok).sum())
        if nb and self.first_bad is None:
            i = int((~ok).flatten().nonzero()[0])
            self.first_bad = (where, i, float(g.flatten()[i]), float(l.flatten()[i]), float(m.flatten()[i]), float(h.flatten()[i]))
        self.bad += nb
        self.ties += int((h != l).sum())
        self.equal += int((g == m).sum())
        self.worst = max(self.worst, float(ratio.nan_to_num(nan=float("inf")).max()) if g.numel() else 0.0)

    def report(self):
        print(f"\n[{self.name}] {self.n} values: worst |kernel - emul(acc)| / B = {self.worst:.3f}, "
              f"bracket holds more than one value: {self.ties / max(self.n, 1):.3e}, "
              f"bit-equal to emul(acc): {self.equal / max(self.n, 1):.6f}")
        assert self.bad == 0, f"{self.name}: {self.bad} values outside the bracket; first (chunk, index, kernel, lo, emul, hi) = {self.first_bad}"


def checked_tiles(n: int, spread: int = 14):
    """The first, the last (ragged) and ``spread`` more spread over the range: on later trips of different CTAs."""
    return sorted(set([0, n - 1] + [round(i * (n - 1) / (spread + 1)) for i in range(1, spread + 1)]))


# ---------------------------------------------------------------------------------------------------------------------
# emulator self-test (CPU): at B = 0 the emulation is one more fp32 implementation of the reference formula
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,lk,ok", [("small", "layers", "out"), ("small", "layers_unsorted", "out_unsorted"),
                                        ("2b", "layers", "out")])
def test_intensity_emulator_matches_reference(name, lk, ok):
    kat = np.load(os.path.join(ROOT, "tests", "golden", "kat_feature.npz"))
    cb0 = torch.from_numpy(kat[f"{name}/cb0"])
    lw = torch.from_numpy(kat[f"{name}/lw"])
    codes = torch.from_numpy(kat[f"{name}/codes"].astype(np.int64))
    centers = torch.from_numpy(kat[f"{name}/centers"]).long()
    layers = [int(l) for l in kat[f"{name}/{lk}"]]
    emu = IntensityEmu(cb0, lw, layers, torch.device("cpu"))
    flat = codes.reshape(-1, codes.shape[-1])
    acc, _ = emu.acc(centers, flat, with_s=False)
    out = emu.out(acc)                                                          # (F, C sorted, T)
    order = [emu.cuts.index(l) for l in layers]
    out = out[:, order]                                                         # (F, len(layers), T)
    Fn = centers.shape[0]
    ref = torch.from_numpy(kat[f"{name}/{ok}"]).reshape(Fn, -1, len(layers)).transpose(1, 2)
    assert float((out.float() - ref.float()).abs().max()) <= ATOL
    sims = fo.codebook_sims(cb0)
    for f in range(Fn):
        exact = fo.intensity_f64(sims, centers[f], flat, lw, layers).T
        steps = fo.intensity_steps(sims, centers[f], flat, lw, layers).T
        assert float((out[f].double() - exact).abs().max()) <= 1e-3
        assert float((out[f].float() - steps.float()).abs().max()) <= ATOL


@pytest.mark.parametrize("case", ["round_fsq_d256", "round_fsq_d512_ml16", "round_fsq_d768_trained", "round_fsq_cbs3"])
def test_decode_emulator_three_passes_matches_exact_decode(golden_small, case):
    from tests import util
    d = util.small_case(golden_small, case)
    m = util.module_from_case(d)
    codes = torch.from_numpy(d["codes_full"].astype(np.int64))
    flat = codes.reshape(-1, codes.shape[-1])
    emu = DecodeEmu(m, 3, d["dec_layers"], min(flat.shape[-1], m.num_quantizers), torch.device("cpu"))
    acc, _ = emu.acc(flat)
    got = emu.out(acc).reshape(d["dec"].shape).numpy()
    assert np.abs(got - d["dec"]).max() <= 2e-5 * np.abs(d["dec"]).max()
    one = DecodeEmu(m, 1, d["dec_layers"], flat.shape[-1], torch.device("cpu"))
    a1, _ = one.acc(flat)
    assert np.abs(one.out(a1).reshape(d["dec"].shape).numpy() - d["dec"]).max() <= 1e-3 * np.abs(d["dec"]).max()


# ---------------------------------------------------------------------------------------------------------------------
# GPU cases
# ---------------------------------------------------------------------------------------------------------------------
def _dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


class _Stub:
    """What intensity_many needs from the model: the codebook and the method name."""
    quantization_method = "round_fsq"

    def __init__(self, cb0, dev):
        self.codebook = torch.nn.Parameter(cb0[None].to(dev), requires_grad=False)


@pytest.fixture(scope="module", autouse=True)
def _file_runtime():
    t0 = time.perf_counter()
    yield
    print(f"\n[test_tc_gemm_gpu] module wall time {time.perf_counter() - t0:.1f} s")


def _round_fsq_cb0():
    from rqae_b200 import RQAE
    return RQAE(dim=16, num_quantizers=1).codebook.data[0].clone()               # the 625-row grid


def _gen(dev, seed):
    return torch.Generator(device=dev).manual_seed(seed)


def _check_intensity(name, out, emu, centers, codes, token_ranges, full_atol=True):
    """Bracket on the given token ranges (every feature and cut); reference-form tolerance on every token."""
    br = Bracket(name)
    for t0, t1 in token_ranges:
        acc, S = emu.acc(centers, codes[t0:t1])
        br.add(out[:, :, t0:t1], *emu.bracket(acc, S), where=(t0, t1))
    if full_atol:
        wc = torch.from_numpy(emu.wc).to(emu.dev).double()[None, :, None]
        T = codes.shape[0]
        worst = 0.0
        for t0 in range(0, T, 4096):
            acc, _ = emu.acc(centers, codes[t0:t0 + 4096], with_s=False)
            worst = max(worst, float((out[:, :, t0:t0 + 4096].double() - acc / wc).abs().max()))
        print(f"[{name}] all {T} tokens: max |kernel - acc / wc| = {worst:.2e}")
        assert worst <= ATOL
    br.report()


@pytest.mark.gpu
def test_intensity_production_shape_with_stagger():
    """F = 513 (5 feature tiles: 3 pairs, the last one single), nq = 1024 with the 14 cuts of scripts/3 (NKB = 70), and
    ceil(4 SMs / 3) + 1 token tiles less a ragged tail: every CTA runs 4-5 units with the start stagger on.  Bracket on
    every feature and cut of 16 token tiles; the whole tensor within ATOL of acc / wc.  The same call twice, on a side
    stream and through the workspace's ``again`` path with another feature set first: bit-identical."""
    from rqae_b200 import _lib
    from rqae_b200.feature import IntensityWorkspace, intensity_many
    dev = _dev()
    sms = _sms()
    Fn, n_pairs = 513, 3
    tiles = -(-4 * sms // 3) + 1
    T = tiles * TOK - 37
    units = tiles * n_pairs
    assert (Fn + 127) // 128 == 5 and units >= 4 * sms and len(SCRIPT3_LAYERS) >= 4     # the stagger runs
    assert units >= 2 * sms and math.gcd(sms, n_pairs) == 1
    cb0 = _round_fsq_cb0()
    lw = (torch.rand(1024, generator=torch.Generator().manual_seed(1)) * 1.5 + 0.25).half()
    model = _Stub(cb0, dev)
    codes = torch.randint(0, 625, (T, 1024), generator=_gen(dev, 2), device=dev, dtype=torch.int16)
    centers = torch.randint(0, 625, (Fn, 1024), generator=_gen(dev, 3), device=dev, dtype=torch.int32)
    centers[7] = codes[123].int()
    out = intensity_many(model, codes, centers, SCRIPT3_LAYERS, layer_weights=lw)
    torch.cuda.synchronize()
    emu = IntensityEmu(cb0, lw, SCRIPT3_LAYERS, dev)
    ranges = [(t * TOK, min(T, (t + 1) * TOK)) for t in checked_tiles(tiles)]
    _check_intensity("intensity 513 x 14 cuts x %d tokens" % T, out, emu, centers, codes, ranges)
    again = intensity_many(model, codes, centers, SCRIPT3_LAYERS, layer_weights=lw)
    assert torch.equal(out, again)
    del again
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        s_out = intensity_many(model, codes, centers, SCRIPT3_LAYERS, layer_weights=lw)
    side.synchronize()
    assert torch.equal(out, s_out)
    del s_out
    ws = IntensityWorkspace()
    assert torch.equal(out, intensity_many(model, codes, centers, SCRIPT3_LAYERS, layer_weights=lw, workspace=ws))
    other = torch.randint(0, 625, (200, 1024), generator=_gen(dev, 4), device=dev, dtype=torch.int32)
    lib = _lib.load()
    n0 = int(lib.rqae_launch_count(0))
    reused = intensity_many(model, codes, other, SCRIPT3_LAYERS, layer_weights=lw, workspace=ws)
    assert int(lib.rqae_launch_count(0)) - n0 == 3                                   # no code copy: the again path ran
    assert torch.equal(reused, intensity_many(model, codes, other, SCRIPT3_LAYERS, layer_weights=lw))


@pytest.mark.gpu
def test_intensity_every_layer_a_cut():
    """Cuts at layers 0..63: every K-block ends a cut, so both accumulators are handed to the epilogue at every step and
    across unit boundaries; F = 600 (3 pairs, the last single), more units than SMs."""
    from rqae_b200.feature import intensity_many
    dev = _dev()
    sms = _sms()
    Fn, n_pairs = 600, 3
    tiles = sms // n_pairs + 7
    T = tiles * TOK - 5
    assert tiles * n_pairs > sms and math.gcd(sms, n_pairs) == 1
    layers = list(range(64))
    cb0 = _round_fsq_cb0()
    lw = (torch.rand(64, generator=torch.Generator().manual_seed(5)) * 1.5 + 0.25).half()
    codes = torch.randint(0, 625, (T, 64), generator=_gen(dev, 6), device=dev, dtype=torch.int16)
    centers = torch.randint(0, 625, (Fn, 64), generator=_gen(dev, 7), device=dev, dtype=torch.int32)
    out = intensity_many(_Stub(cb0, dev), codes, centers, layers, layer_weights=lw)
    torch.cuda.synchronize()
    emu = IntensityEmu(cb0, lw, layers, dev)
    ranges = [(t * TOK, min(T, (t + 1) * TOK)) for t in checked_tiles(tiles)]
    _check_intensity("intensity 64 cuts", out, emu, centers, codes, ranges)


@pytest.mark.gpu
def test_intensity_deepest_schedule_and_limits():
    """NKB = 200 exactly (one cut at layer 3199) with more units than SMs; NKB = 201 and 65 cuts are refused."""
    from rqae_b200.feature import intensity_many
    dev = _dev()
    sms = _sms()
    tiles = sms + 2
    T = tiles * TOK - 100
    cb0 = _round_fsq_cb0()
    lw = (torch.rand(3216, generator=torch.Generator().manual_seed(8)) * 1.5 + 0.25).half()
    codes = torch.randint(0, 625, (T, 3200), generator=_gen(dev, 9), device=dev, dtype=torch.int16)
    centers = torch.randint(0, 625, (129, 3200), generator=_gen(dev, 10), device=dev, dtype=torch.int32)
    model = _Stub(cb0, dev)
    out = intensity_many(model, codes, centers, [3199], layer_weights=lw)
    torch.cuda.synchronize()
    emu = IntensityEmu(cb0, lw, [3199], dev)
    assert emu.nkb == [200] and tiles > sms
    ranges = [(t * TOK, min(T, (t + 1) * TOK)) for t in checked_tiles(tiles)]
    _check_intensity("intensity NKB = 200", out, emu, centers, codes, ranges)
    wide = torch.zeros(2, 3216, dtype=torch.int16, device=dev)
    with pytest.raises(NotImplementedError):
        intensity_many(model, wide, wide[:1], [3215], layer_weights=lw)             # 201 K-blocks
    with pytest.raises(NotImplementedError):
        intensity_many(model, wide, wide[:1], list(range(65)), layer_weights=lw)    # 65 cuts


@pytest.mark.gpu
def test_intensity_codebook_sizes():
    """K = 639 (the largest lookup table, random codebook) with more units than SMs; K = 640 is refused; K = 81 (codebook
    size 3) is accepted."""
    from rqae_b200.feature import intensity_many
    dev = _dev()
    sms = _sms()
    g = torch.Generator().manual_seed(12)
    lw = (torch.rand(100, generator=g) * 1.5 + 0.25).half()
    layers = [9, 40, 99]
    tiles = sms + 9
    T = tiles * TOK - 100
    for K, T_k, checked in ((639, T, checked_tiles(tiles)), (81, 700, None)):
        cb0 = torch.randn(K, 4, generator=g)
        codes = torch.randint(0, K, (T_k, 100), generator=_gen(dev, K), device=dev, dtype=torch.int16)
        codes[:, 7] = K - 1
        centers = torch.randint(0, K, (129, 100), generator=_gen(dev, K + 1), device=dev, dtype=torch.int32)
        centers[:, 3] = K - 1
        out = intensity_many(_Stub(cb0, dev), codes, centers, layers, layer_weights=lw)
        torch.cuda.synchronize()
        emu = IntensityEmu(cb0, lw, layers, dev)
        ranges = [(0, T_k)] if checked is None else [(t * TOK, min(T_k, (t + 1) * TOK)) for t in checked]
        _check_intensity(f"intensity K = {K}", out, emu, centers, codes, ranges)
    cb0 = torch.randn(640, 4, generator=g)
    with pytest.raises(RuntimeError, match="unsupported"):
        intensity_many(_Stub(cb0, dev), codes[:10], centers, layers, layer_weights=lw)


@pytest.mark.gpu
@pytest.mark.parametrize("Fn", [1, 33, 129])
@pytest.mark.parametrize("T", [1, 255, 257])
def test_intensity_ragged_sizes_write_nothing_outside(Fn, T):
    """Ragged feature and token counts into ``out=buf[:F]`` of a NaN-filled buffer with a spare row and 256 spare
    columns: every value inside the bracket, row F and every column >= T_pad still NaN."""
    from rqae_b200.feature import intensity_many
    dev = _dev()
    layers = [0, 17, 63]
    cb0 = _round_fsq_cb0()
    lw = (torch.rand(64, generator=torch.Generator().manual_seed(Fn + T)) * 1.5 + 0.25).half()
    codes = torch.randint(0, 625, (T, 64), generator=_gen(dev, T), device=dev, dtype=torch.int16)
    centers = torch.randint(0, 625, (Fn, 64), generator=_gen(dev, Fn), device=dev, dtype=torch.int32)
    T_pad = (T + TOK - 1) // TOK * TOK
    buf = torch.full((Fn + 1, len(layers), T_pad + 256), float("nan"), dtype=torch.float16, device=dev)
    out = intensity_many(_Stub(cb0, dev), codes, centers, layers, layer_weights=lw, out=buf[:Fn])
    torch.cuda.synchronize()
    assert out.data_ptr() == buf.data_ptr()
    assert bool(buf[Fn].isnan().all()) and bool(buf[:, :, T_pad:].isnan().all())
    _check_intensity(f"intensity F = {Fn}, T = {T}", out, IntensityEmu(cb0, lw, layers, dev), centers, codes, [(0, T)])


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["int16_vector", "int16_scalar", "int32", "int64"])
def test_intensity_code_paths_and_out_of_range_codes(path):
    """Every branch of int_transpose_kernel: int16 with 16-byte loads (row stride a multiple of 8, aligned), int16 through
    the scalar path (a view one element into a wider tensor), int32 and int64; L = 101 (the last 32-layer block always
    scalar); negative int16, int32 equal to K, int64 2^32 + 5 and -1, centers outside [0, K): all contribute zero."""
    from rqae_b200.feature import intensity_many
    dev = _dev()
    layers = [5, 40, 100]
    T, nq, K = 3 * TOK - 9, 104, 625
    cb0 = _round_fsq_cb0()
    lw = (torch.rand(nq, generator=torch.Generator().manual_seed(14)) * 1.5 + 0.25).half()
    base = torch.randint(0, K, (T, nq), generator=_gen(dev, 15), device=dev, dtype=torch.int64)
    base[:, 11] = K - 1
    centers = torch.randint(0, K, (40, nq), generator=_gen(dev, 16), device=dev, dtype=torch.int32)
    centers[1, 2], centers[2, 50], centers[3, 99] = -1, K, 1000000
    if path.startswith("int16"):
        base[3, 4], base[7, 0], base[9, 100], base[300, 60] = -3, -32768, 32767, K
        if path == "int16_vector":
            codes = base.to(torch.int16)
            assert codes.stride(0) % 8 == 0 and codes.data_ptr() % 16 == 0
        else:
            big = torch.zeros(T, nq + 8, dtype=torch.int16, device=dev)
            big[:, 1:nq + 1] = base
            codes = big[:, 1:nq + 1]
            assert codes.data_ptr() % 16 != 0
    elif path == "int32":
        base[3, 4], base[8, 33], base[500, 100] = K, K, -7
        codes = base.to(torch.int32)
    else:
        base[3, 4], base[8, 33], base[500, 100], base[600, 0] = 2 ** 32 + 5, -1, 2 ** 40, K
        codes = base
    out = intensity_many(_Stub(cb0, dev), codes, centers, layers, layer_weights=lw)
    torch.cuda.synchronize()
    _check_intensity(f"intensity codes {path}", out, IntensityEmu(cb0, lw, layers, dev), centers, codes, [(0, T)])


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16", "f16x3"])
@pytest.mark.parametrize("holes", [False, True])
def test_decode_tc_many_units(precision, holes):
    """D = 600 (5 tiles, the last partial: 3 pairs), nq = 1024 (NKB = 64 / 192), 2 SMs + 1 token tiles less a ragged tail
    (units >= 2 SMs); a ``layers=`` selection with holes; codes -1 and -625 take the python-style rows K - 1 and 0, as in
    the bit-exact decode, and 625 and -626 the zero row.  Bracket on every dimension of 16 token tiles; the whole output
    within the stated relative error of the bit-exact decode (tests/test_parity_gpu.py).  Before the decode wrapped
    negative codes, the -1 made this error 1.2e-2 of max |q| in both precisions."""
    from rqae_b200 import RQAE
    dev = _dev()
    sms = _sms()
    D, n_pairs = 600, 3
    tiles = -(-2 * sms // n_pairs) + 1
    T = tiles * TOK - 44
    assert tiles * n_pairs >= 2 * sms and math.gcd(sms, n_pairs) == 1
    torch.manual_seed(17)
    m = RQAE(dim=D, num_quantizers=1024).eval().to(dev)
    codes = torch.randint(0, 625, (T, 1024), generator=_gen(dev, 18), device=dev, dtype=torch.int16)
    codes[5, 9], codes[6, 1000], codes[7, 3], codes[8, 4] = -1, 625, -625, -626   # last row, zero, row 0, zero
    layers = [l for l in range(1024) if l % 7 != 3 and not 200 <= l < 260] if holes else None
    passes = 1 if precision == "f16" else 3
    q = m.decode(codes, layers=layers, precision=precision)
    exact = m.decode(codes, layers=layers)
    torch.cuda.synchronize()
    emu = DecodeEmu(m, passes, layers, 1024, dev)
    assert emu.nkb == passes * 64
    br = Bracket(f"decode {precision}{' with holes' if holes else ''}")
    for t in checked_tiles(tiles):
        t0, t1 = t * TOK, min(T, (t + 1) * TOK)
        acc, S = emu.acc(codes[t0:t1])
        br.add(q[t0:t1], *emu.bracket(acc, S), where=(t0, t1))
    rel = float((q - exact).abs().max()) / float(exact.abs().max())
    print(f"[decode {precision}] all {T} tokens: max |tc - exact| / max |exact| = {rel:.2e}")
    assert rel <= (1e-3 if precision == "f16" else 5e-5)
    br.report()


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode,S,Sq", [("projected", 127, 128), ("original", 128, 1), ("original", 127, 128),
                                       ("projected", 128, 128)])
def test_search_tc_many_units(mode, S, Sq):
    """4 SMs + 3 sequences (odd: the last unit holds one), S = 127 (a padding column) or 128, nq = 150 with range ends that
    are not multiples of 8, 1 or 128 query positions.  Bracket on every (cut, query position, sequence); sequence 4 is
    built so that, for query position 0, every position's prefix is negative.  find_examples(precision="tc") on the
    same store reports the exact accumulation rows bit for bit."""
    from rqae_b200 import RQAE
    from rqae_b200.search import IntensityEngine
    dev = _dev()
    sms = _sms()
    n_seq, nq = 4 * sms + 3, 150
    units = (n_seq + 1) // 2
    assert n_seq % 2 == 1 and units >= 2 * sms
    layers = [3, 13, 22, 37, 64, 101, 150]
    torch.manual_seed(19)
    model = RQAE(dim=256, num_quantizers=nq).eval().to(dev)
    K = model.codebook.shape[1]
    codes = torch.randint(0, K, (n_seq, S, nq), generator=_gen(dev, 20), device=dev, dtype=torch.int32)
    codes[1, 2, 3], codes[2, 0, 149] = -1, K
    query = torch.randint(0, K, (Sq, nq), generator=_gen(dev, 21), device=dev, dtype=torch.int32)
    tc = IntensityEngine(model, codes.to(torch.int16), mode=mode, precision="tc")
    # the code with the most negative factor product against query position 0, at every layer of sequence 4
    dots = torch.einsum("lj,lkj->lk", tc._utab[torch.arange(nq, device=dev), query[0].long()].double(), tc._vtab[:nq].double())
    dots[:, K:] = float("inf")
    codes[4] = dots.argmin(dim=1).int()[None, :]
    tc = IntensityEngine(model, codes.to(torch.int16), mode=mode, precision="tc")
    q = tc._query(None, query, max(layers))
    got = tc.maxima_tc(q, layers)                                                   # (C, Sq, N)
    torch.cuda.synchronize()
    br = Bracket(f"search-tc {mode}, S = {S}, Sq = {Sq}")
    for n0 in range(0, n_seq, 64):
        sl = slice(n0, min(n_seq, n0 + 64))
        lo, mid, hi, mx = search_emu(tc, q, layers, sl)
        if n0 == 0:
            assert bool((mx[:, 0, 4] < 0).all())        # the padding column (prefix 0) must stay out of this maximum
        br.add(got[:, :, sl], lo, mid, hi, where=n0)
    br.report()
    exact = IntensityEngine(model, codes.to(torch.int16), mode=mode)
    accs = [a.clone() for a, _ in exact.accumulate(q, layers)]
    qpos = torch.arange(Sq, device=dev).unsqueeze(-1)
    res = list(tc.find_examples(activation=query.cpu(), top_examples=30, middle_examples=10, bottom_examples=10,
                                layers=layers))
    assert [l for _, l in res] == layers
    for (r, _), acc in zip(res, accs):
        for part in ("top", "middle", "bottom"):
            idx = r[part]["indices"].long().to(dev)
            assert torch.equal(r[part]["intensities"].to(dev), acc[idx, :, qpos]), part


# ---------------------------------------------------------------------------------------------------------------------
# IntensityWorkspace reuse
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_workspace_not_reused_for_a_new_tensor_at_a_freed_address():
    """A code tensor is freed and a new one of the same shape lands at its address with the same ``_version``: the
    workspace must not take it for the old one."""
    from rqae_b200.feature import IntensityWorkspace, intensity_many
    dev = _dev()
    cb0 = _round_fsq_cb0()
    layers = [3, 20, 47]
    lw = (torch.rand(48, generator=torch.Generator().manual_seed(22)) * 1.5 + 0.25).half()
    centers = torch.randint(0, 625, (30, 48), generator=torch.Generator().manual_seed(23), dtype=torch.int32)
    first = torch.randint(0, 625, (600, 48), generator=torch.Generator().manual_seed(24)).to(torch.int16)
    second = torch.randint(0, 625, (600, 48), generator=torch.Generator().manual_seed(25)).to(torch.int16)
    model = _Stub(cb0, dev)
    ws = IntensityWorkspace()
    a = first.to(dev)
    ptr, ver = a.data_ptr(), a._version
    intensity_many(model, a, centers, layers, layer_weights=lw, workspace=ws)
    torch.cuda.synchronize()
    del a
    b = second.to(dev)
    assert b.data_ptr() == ptr and b._version == ver          # the coincidence this test is about
    got = intensity_many(model, b, centers, layers, layer_weights=lw, workspace=ws)
    assert torch.equal(got, intensity_many(model, b, centers, layers, layer_weights=lw))


@pytest.mark.gpu
def test_workspace_not_reused_after_an_in_place_change_of_a_copied_store():
    """A non-contiguous code store (copied by intensity_many on every call) changed in place between two calls: the
    second call must see the new codes."""
    from rqae_b200.feature import IntensityWorkspace, intensity_many
    dev = _dev()
    cb0 = _round_fsq_cb0()
    layers = [3, 20, 47]
    lw = (torch.rand(48, generator=torch.Generator().manual_seed(26)) * 1.5 + 0.25).half()
    centers = torch.randint(0, 625, (30, 48), generator=torch.Generator().manual_seed(27), dtype=torch.int32)
    big = torch.randint(0, 625, (600, 96), generator=_gen(dev, 28), device=dev, dtype=torch.int16)
    store = big[:, ::2]
    assert not store.is_contiguous()
    model = _Stub(cb0, dev)
    ws = IntensityWorkspace()
    before = intensity_many(model, store, centers, layers, layer_weights=lw, workspace=ws).clone()
    store.copy_(torch.randint(0, 625, (600, 48), generator=_gen(dev, 29), device=dev, dtype=torch.int16))
    got = intensity_many(model, store, centers, layers, layer_weights=lw, workspace=ws)
    want = intensity_many(model, store, centers, layers, layer_weights=lw)
    assert not torch.equal(want, before)
    assert torch.equal(got, want)
