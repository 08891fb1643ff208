"""The bit-exact feature intensities (``intensity_many(..., precision="exact")``, ``rqae_intensity_exact_f16``).

Every GPU case compares bit patterns: against outputs of the unmodified reference (tests/golden/kat_feature.npz,
tests/golden/kat_mining.npz) and against ``oracle.feature_oracle.intensity_steps``, which writes out every rounding of
the reference.  The argument checks at the end run without a GPU: the library validates before any CUDA call."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import feature_oracle as fo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ATOL = 2e-3    # the tensor-core path's tolerance (tests/test_feature_gpu.py)
K = 625


def _dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _bits(t: torch.Tensor) -> torch.Tensor:
    return t.detach().cpu().contiguous().view(torch.int16)


def _same_bits(a, b) -> bool:
    return a.shape == b.shape and torch.equal(_bits(a), _bits(b))


class _Stub:
    """What intensity_many needs from the model: the codebook and the method name."""
    quantization_method = "round_fsq"

    def __init__(self, cb0, dev):
        self.codebook = torch.nn.Parameter(cb0[None].to(dev), requires_grad=False)


def _round_fsq_stub(dev):
    from rqae_b200.model import _fsq_grid
    return _Stub(_fsq_grid(5, 4, True), dev)


def _oracle(sims, center, codes, w, layers):
    """intensity_steps with the kernel's indexing rule: codes in [-K, 0) wrap, codes outside [-K, K) read an appended
    all-+0 row / column (the reference raises there).  codes (T, nq) -> (len(layers), T)."""
    k = sims.shape[0]
    ext = torch.zeros(k + 1, k + 1, dtype=torch.float16)
    ext[:k, :k] = sims

    def row(c):
        c = c.long()
        c = torch.where(c < 0, c + k, c)
        return torch.where((c >= 0) & (c < k), c, torch.full_like(c, k))
    return fo.intensity_steps(ext, row(center), row(codes), w, layers).T


# ---------------------------------------------------------------------------------------------------------------------
# 1. the reference's goldens
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.int16, torch.int32, torch.int64])
@pytest.mark.parametrize("name,lk,ok", [("small", "layers", "out"), ("small", "layers_unsorted", "out_unsorted"),
                                        ("2b", "layers", "out")])
def test_exact_equals_reference_golden(name, lk, ok, dtype):
    from rqae_b200.feature import intensity_many
    kat = np.load(os.path.join(ROOT, "tests", "golden", "kat_feature.npz"))
    dev = _dev()
    codes = torch.from_numpy(kat[f"{name}/codes"].astype(np.int64))
    centers = torch.from_numpy(kat[f"{name}/centers"])
    layers = [int(l) for l in kat[f"{name}/{lk}"]]
    out = intensity_many(_Stub(torch.from_numpy(kat[f"{name}/cb0"]), dev), codes.to(dev).to(dtype), centers, layers,
                         layer_weights=torch.from_numpy(kat[f"{name}/lw"]), precision="exact")
    ref = torch.from_numpy(kat[f"{name}/{ok}"])
    ref = ref.reshape(centers.shape[0], -1, len(layers)).transpose(1, 2)           # (F, C, T)
    assert out.dtype == torch.float16 and _same_bits(out, ref)


# ---------------------------------------------------------------------------------------------------------------------
# 2. upstream's mined activation rows (scripts/3_make_rqae_features.py)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("top_k", [7, 100])
def test_exact_mining_equals_upstream_rows(top_k):
    from rqae_b200.feature import FeatureHelper, RQAEFeature, intensity_many
    kat = np.load(os.path.join(ROOT, "tests", "golden", "kat_mining.npz"))
    dev = _dev()
    cb0 = torch.from_numpy(kat["cb0"])
    model = _Stub(cb0, dev)
    codes = torch.from_numpy(kat["codes"].astype(np.int64))
    N, S, _ = codes.shape
    layers = [int(l) for l in kat["layers"]]
    lw = torch.from_numpy(kat["lw"])
    centers = torch.from_numpy(kat["centers"])
    feats = []
    for c in kat["centers"]:
        f = RQAEFeature(num_quantizers=64, dim=4, center=c, layers=layers)
        f.rqae, f.layer_weights = model, lw
        feats.append(f)
    helper = FeatureHelper(torch.zeros(N, S, dtype=torch.int64), list(range(N)), codes.to(dev).to(torch.int16))
    many = helper.get_activations_many(feats, top_k=top_k, precision="exact")
    inten = intensity_many(model, helper.indices, centers, layers, layer_weights=lw, precision="exact").cpu()
    sims = fo.codebook_sims(cb0)
    flat = codes.reshape(N * S, -1)
    windows = 0
    for fi, acts in enumerate(many):
        ref = fo.intensity(sims, centers[fi], flat, lw, layers)                         # (T, C): the reference's calls
        assert _same_bits(inten[fi].T, ref)
        want = fo.get_activations(ref, layers, top_k, S, stable=True)
        for j, l in enumerate(layers):
            seqs, rows = want[l]
            assert [a["text"] for a in acts[l]] == seqs, (fi, l)
            got = np.stack([a["activations"] for a in acts[l]])
            assert got.dtype == np.float16 and np.array_equal(got.view(np.uint16), rows.view(np.uint16)), (fi, l)
            # every sequence the unmodified script wrote: its row of exact intensities, bit for bit
            gold_seqs = [int(s) for s in kat[f"f{fi}/k{top_k}/{l}/sequences"]]
            gold_rows = kat[f"f{fi}/k{top_k}/{l}/activations"]
            mine = inten[fi, j].reshape(N, S)[gold_seqs].numpy()
            assert np.array_equal(mine.view(np.uint16), gold_rows.view(np.uint16)), (fi, l)
            windows += 1
    assert windows == 20
    one = helper.get_activations(feats[0], top_k=top_k, precision="exact")
    assert [a["text"] for a in one[layers[-1]]] == [a["text"] for a in many[0][layers[-1]]]


# ---------------------------------------------------------------------------------------------------------------------
# 3. random shapes against intensity_steps
# ---------------------------------------------------------------------------------------------------------------------
def _random_case(F, T, nq, seed, dtype, wild=True):
    g = torch.Generator().manual_seed(seed)
    codes = torch.randint(0, K, (T, nq), generator=g)
    centers = torch.randint(0, K, (F, nq), generator=g)
    centers[0, :5] = 312                                         # the zero codeword: a row of +0 (other rows hold -0)
    if wild:
        neg = torch.rand(T, nq, generator=g) < 0.01
        codes[neg] = torch.randint(-K, 0, (int(neg.sum()),), generator=g)            # wrap to code + K
        bad = torch.rand(T, nq, generator=g) < 0.002
        big = 32000 if dtype == torch.int16 else (1 << 40 if dtype == torch.int64 else 1 << 30)
        codes[bad] = torch.tensor([K, -K - 1, big, -big])[torch.randint(0, 4, (int(bad.sum()),), generator=g)]
        centers[-1, 1::7] = torch.randint(-K, 0, centers[-1, 1::7].shape, generator=g)
        centers[-1, 3::11] = K + 3
    lw = (torch.rand(nq, generator=g) * 2 + 13).half()
    return codes.to(dtype), centers, lw


@pytest.mark.gpu
@pytest.mark.parametrize("F,T,nq,layers,dtype", [
    (1, 1000, 64, [0, 5, 13, 63], torch.int16),
    (7, 40003, 160, [0, 7, 8, 9, 100, 159], torch.int32),
    (9, 1000, 160, list(range(160)), torch.int64),                # every layer a cut: more than the GEMM's 64
    (300, 1000, 64, [63, 0, 17, 17, 40], torch.int16),            # unsorted and repeated, as the reference allows
])
def test_exact_equals_intensity_steps(F, T, nq, layers, dtype):
    from rqae_b200.feature import intensity_many
    dev = _dev()
    m = _round_fsq_stub(dev)
    codes, centers, lw = _random_case(F, T, nq, F * 1000 + nq, dtype)
    out = intensity_many(m, codes.to(dev), centers, layers, layer_weights=lw, precision="exact").cpu()
    assert out.shape == (F, len(layers), T)
    sims = fo.codebook_sims(m.codebook.data[0].cpu())
    for f in sorted({0, 1, F // 2, F - 1} & set(range(F))):
        assert _same_bits(out[f], _oracle(sims, centers[f], codes, lw, layers)), f
    if 0 in layers:   # feature 0 is centred on the zero codeword at layer 0: +-0 products, +0 intensities
        assert int(_bits(out[0, layers.index(0)]).ne(0).sum()) == 0


@pytest.mark.gpu
def test_exact_production_depth_many_units():
    """nq = 1024, the 14 cuts of scripts/3:178, more (token tile, feature group) units than the device has SMs."""
    from rqae_b200.feature import intensity_many, SCRIPT3_LAYERS
    dev = _dev()
    F, T = 300, 40003
    units = (T + 2047) // 2048 * ((F + 7) // 8)
    assert units > torch.cuda.get_device_properties(dev).multi_processor_count
    m = _round_fsq_stub(dev)
    codes, centers, lw = _random_case(F, T, 1024, 5, torch.int16)
    out = intensity_many(m, codes.to(dev), centers, SCRIPT3_LAYERS, layer_weights=lw, precision="exact").cpu()
    sims = fo.codebook_sims(m.codebook.data[0].cpu())
    for f in (0, 7, 8, 151, 299):
        assert _same_bits(out[f], _oracle(sims, centers[f], codes, lw, SCRIPT3_LAYERS)), f


@pytest.mark.gpu
def test_exact_layer0_negative_zero_gives_positive_zero():
    """A cut at layer 0 on a (-0 table entry) pair: the running sum starts at +0, so the result is +0, not -0."""
    from rqae_b200.feature import intensity_many
    dev = _dev()
    m = _round_fsq_stub(dev)
    sims = fo.codebook_sims(m.codebook.data[0].cpu())
    pairs = (sims.view(torch.int16) == -32768).nonzero()                             # (center code, token code)
    assert pairs.numel() > 0
    r = int(pairs[:, 0].mode().values)
    neg = pairs[pairs[:, 0] == r, 1]
    codes = torch.zeros(neg.numel(), 4, dtype=torch.int32)
    codes[:, 0] = neg.int()
    centers = torch.full((1, 4), r, dtype=torch.int32)
    lw = torch.tensor([1.5, 2.0, 1.0, 1.0]).half()
    out = intensity_many(m, codes.to(dev), centers, [0, 3], layer_weights=lw, precision="exact").cpu()
    assert int(_bits(out[0, 0]).eq(0).sum()) == neg.numel()                         # all +0
    assert _same_bits(out[0], _oracle(sims, centers[0], codes, lw, [0, 3]))


@pytest.mark.gpu
def test_rqae_feature_intensity_all_layers():
    """RQAEFeature.intensity(codes, layers=range(nq), precision="exact"), as the reference allows (no 64-cut limit)."""
    from rqae_b200 import RQAEFeature
    dev = _dev()
    m = _round_fsq_stub(dev)
    codes, centers, lw = _random_case(1, 3 * 77, 96, 3, torch.int64, wild=False)
    f = RQAEFeature(num_quantizers=96, dim=4, center=centers[0].numpy(), layers=[95])
    f.rqae, f.layer_weights = m, lw
    got = f.intensity(codes.reshape(3, 77, 96).to(dev), layers=range(96), precision="exact")
    assert got.shape == (3, 77, 96)
    sims = fo.codebook_sims(m.codebook.data[0].cpu())
    ref = fo.intensity(sims, centers[0], codes.reshape(3, 77, 96), lw, list(range(96)))
    assert _same_bits(got, ref)
    with pytest.raises(ValueError):
        f.intensity(codes.to(dev), precision="bogus")


# ---------------------------------------------------------------------------------------------------------------------
# 4. launches, streams, buffers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_exact_one_launch_repeatable_on_any_stream():
    from rqae_b200 import _lib
    from rqae_b200.feature import intensity_many
    dev = _dev()
    lib = _lib.load()
    m = _round_fsq_stub(dev)
    codes, centers, lw = _random_case(20, 5000, 128, 9, torch.int16)
    codes = codes.to(dev)
    layers = [1, 30, 64, 127]
    a = intensity_many(m, codes, centers, layers, layer_weights=lw, precision="exact").clone()   # table cached here
    n0 = int(lib.rqae_launch_count(0))
    b = intensity_many(m, codes, centers, layers, layer_weights=lw, precision="exact").clone()
    assert int(lib.rqae_launch_count(0)) - n0 == 1                                  # header: one launch per call
    s = torch.cuda.Stream(dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        c = intensity_many(m, codes, centers, layers, layer_weights=lw, precision="exact").clone()
    torch.cuda.current_stream(dev).wait_stream(s)
    buf = torch.full((20, 4, 5000), float("nan"), dtype=torch.float16, device=dev)
    d = intensity_many(m, codes, centers, layers, layer_weights=lw, out=buf, precision="exact")
    assert d.data_ptr() == buf.data_ptr()
    d = intensity_many(m, codes, centers, layers, layer_weights=lw, out=buf, precision="exact")
    for x in (b, c, d):
        assert _same_bits(a, x)
    n0 = int(lib.rqae_launch_count(0))
    e = intensity_many(m, codes[:0], centers, layers, layer_weights=lw, precision="exact")
    assert e.shape == (20, 4, 0) and int(lib.rqae_launch_count(0)) - n0 == 0


# ---------------------------------------------------------------------------------------------------------------------
# 5. agrees with the tensor-core path
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_exact_within_tolerance_of_gemm():
    from rqae_b200.feature import intensity_many
    kat = np.load(os.path.join(ROOT, "tests", "golden", "kat_feature.npz"))
    dev = _dev()
    m = _Stub(torch.from_numpy(kat["2b/cb0"]), dev)
    codes = torch.from_numpy(kat["2b/codes"].astype(np.int64)).to(dev)
    centers = torch.from_numpy(kat["2b/centers"])
    layers = [int(l) for l in kat["2b/layers"]]
    lw = torch.from_numpy(kat["2b/lw"])
    ex = intensity_many(m, codes, centers, layers, layer_weights=lw, precision="exact").float()
    tc = intensity_many(m, codes, centers, layers, layer_weights=lw).float()
    assert float((ex - tc).abs().max()) <= ATOL


# ---------------------------------------------------------------------------------------------------------------------
# 6. argument validation (no GPU: the library checks its arguments before any CUDA call)
# ---------------------------------------------------------------------------------------------------------------------
def _call(**kw):
    from rqae_b200 import _lib
    a = dict(sims=16, K=625, codes=16, code_dtype=0, code_stride=1024, n_tokens=100, centers=16, center_stride=1024,
             n_features=3, w=16, cuts=[2, 4, 1023], out=1024, out_stride=104)
    a.update(kw)
    cuts = np.asarray(a["cuts"] if a["cuts"] is not None else [], dtype=np.int32)
    cp = None if a["cuts"] is None else cuts.ctypes.data
    return _lib.load().rqae_intensity_exact_f16(a["sims"], a["K"], a["codes"], a["code_dtype"], a["code_stride"],
                                                a["n_tokens"], a["centers"], a["center_stride"], a["n_features"], a["w"],
                                                cp, len(cuts) if a["cuts"] is not None else 0, a["out"],
                                                a["out_stride"], None)


@pytest.mark.parametrize("kw,rc", [
    (dict(sims=None), 1), (dict(codes=None), 1), (dict(centers=None), 1), (dict(w=None), 1), (dict(out=None), 1),
    (dict(cuts=None), 1), (dict(code_dtype=3), 1), (dict(code_dtype=-1), 1), (dict(K=0), 1), (dict(K=-5), 1),
    (dict(K=640), 2), (dict(K=639, n_tokens=0), 0),
    (dict(cuts=[4, 2]), 1), (dict(cuts=[2, 2]), 1), (dict(cuts=[-1, 3]), 1), (dict(cuts=[]), 1),
    (dict(cuts=[0, 4096], code_stride=5000, center_stride=5000), 2),
    (dict(cuts=[0, 4095], code_stride=4096, center_stride=4096, n_tokens=0), 0),
    (dict(code_stride=1023), 1), (dict(center_stride=1023), 1),
    (dict(out_stride=96), 1), (dict(out_stride=100, n_tokens=100), 1), (dict(out_stride=108), 1), (dict(out=1032), 1),
    (dict(out_stride=100, n_tokens=97), 1), (dict(out_stride=104, n_tokens=97, n_features=0), 0),
    (dict(n_tokens=0), 0), (dict(n_features=0), 0), (dict(n_features=-1), 1), (dict(n_tokens=-1), 1),
    (dict(cuts=list(range(200)), n_tokens=0), 0),                                  # no 64-cut limit
])
def test_exact_argument_validation(kw, rc):
    assert _call(**kw) == rc


def test_unknown_precision_raises_before_the_gpu():
    from rqae_b200.feature import intensity_many
    with pytest.raises(ValueError):
        intensity_many(_Stub(torch.zeros(625, 4), torch.device("cpu")), torch.zeros(4, 8, dtype=torch.int16),
                       torch.zeros(1, 8, dtype=torch.int32), [3], precision="bogus")


def test_binding_declared():
    from rqae_b200 import _lib
    assert "rqae_intensity_exact_f16" in _lib.SYMBOLS
    assert hasattr(ctypes.CDLL(_lib.LIB_PATH), "rqae_intensity_exact_f16")
