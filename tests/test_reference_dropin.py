"""``rqae_b200.RQAE`` as a drop-in for the reference class (SURVEY 8b: "rqae/feature.py and
scripts/3_make_rqae_features.py work unchanged").

The reference callers read ``codebook_sims``, ``layers[l][1].weight``, ``num_quantizers``, ``codebook_dim``,
``subfeature_sims`` and ``layer_norms`` of the model object and the reference's state-dict layout.  Here the new
class is built from the same seeds as the reference models behind the committed golden vectors, and what those callers
read from it is compared with what the UNMODIFIED reference produced (tests/golden/make_golden*.py):

  kat_small.npz    constructor weights of seven reference configurations (make_golden.py ``small_case``)
  kat_feature.npz  ``RQAEFeature.from_quantizer(RQAE(dim=64, num_quantizers=64)).intensity`` of the reference
  kat_mining.npz   ``FeatureHelper.get_activations`` of scripts/3 on the same reference model
  kat_search.npz   the server's engine table ``subfeature_sims * layer_norms`` (demo/server/server.py:111)

The reference's own arithmetic after the model attributes is replayed by the oracle ports (oracle/feature_oracle.py),
which tests/test_feature_oracle.py holds bit-identical to the same golden files.  Nothing here touches a GPU."""
import os

import numpy as np
import torch

from oracle import feature_oracle as fo
from tests import util

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# make_golden.py small_case(): constructor arguments and seed of every case whose weights are the constructor's own
# (round_fsq_d768_trained overwrites them after construction)
SMALL_CONSTRUCTORS = {
    "round_fsq_d256": (0, dict(dim=256, num_quantizers=8, quantization_method="round_fsq")),
    "round_fsq_d256_zero": (1, dict(dim=256, num_quantizers=8, quantization_method="round_fsq")),
    "round_fsq_d512_ml16": (2, dict(dim=512, num_quantizers=32, quantization_method="round_fsq")),
    "fsq_d384": (3, dict(dim=384, num_quantizers=12, quantization_method="fsq")),
    "vq_d256": (4, dict(dim=256, num_quantizers=10, quantization_method="vq", codebook_size=64)),
    "round_fsq_d200_ragged": (5, dict(dim=200, num_quantizers=6, quantization_method="round_fsq")),
    "round_fsq_cbs3": (7, dict(dim=128, num_quantizers=5, quantization_method="round_fsq", codebook_size=3)),
}


def _load(name):
    return np.load(os.path.join(GOLDEN, name))


def _new(seed, **kw):
    from rqae_b200 import RQAE
    torch.manual_seed(seed)
    return RQAE(**kw).eval()


def _reference_reads(model):
    """What RQAEFeature.from_quantizer -> load_model (rqae/feature.py:95-99) reads of the model: the fp16 table of
    codebook similarities and the per-layer weights from layers[l][1].weight."""
    w_out = torch.stack([layer[1].weight.detach() for layer in model.layers])
    return model.codebook_sims, fo.layer_weights(w_out)


def _reference_keys(nq):
    keys = ["codebook", "codebook_counts"]
    for l in range(nq):
        keys += [f"layers.{l}.0.weight", f"layers.{l}.0.bias", f"layers.{l}.1.weight", f"layers.{l}.1.bias"]
    return keys


def test_reference_state_dict_loads_strict_both_ways():
    """Same seed, same parameters as the reference constructor (same RNG order), for every quantization method; the
    reference's state dict loads strictly into the new class and the new class's state dict has the reference's keys
    in the reference's order."""
    g = _load("kat_small.npz")
    for name, (seed, kw) in SMALL_CONSTRUCTORS.items():
        new = _new(seed, **kw)
        ref = util.small_case(g, name)
        got = util.stacked_from_module(new)
        for k in ("w_in", "b_in", "w_out", "b_out", "codebook"):
            assert np.array_equal(getattr(got, k).numpy(), ref[k]), (name, k)
        assert list(new.state_dict().keys()) == _reference_keys(kw["num_quantizers"]), name
        back = util.module_from_case(ref)                    # the reference's layout, loaded with strict=True
        back.load_state_dict(new.state_dict(), strict=True)
        for (k, a), (_, b) in zip(back.state_dict().items(), new.state_dict().items()):
            assert torch.equal(a, b), (name, k)


def test_reference_rqaefeature_runs_on_new_class_and_equals_reference_class():
    """rqae/feature.py:95-136: from_quantizer -> load_model (layer weights from layers[l][1].weight) ->
    intensity (gather from codebook_sims), fed by the new class, equals the reference's intensities bit for bit."""
    from rqae_b200 import RQAEFeature
    k = _load("kat_feature.npz")
    new = _new(0, dim=64, num_quantizers=64)
    assert new.num_quantizers == 64 and new.codebook_dim == 4
    assert np.array_equal(new.codebook.data[0].numpy(), k["small/cb0"])
    sims, lw = _reference_reads(new)
    assert torch.equal(sims, fo.codebook_sims(torch.from_numpy(k["small/cb0"])))
    assert torch.equal(lw, torch.from_numpy(k["small/lw"]))
    codes = torch.from_numpy(k["small/codes"].astype(np.int64))
    centers = torch.from_numpy(k["small/centers"])
    for lk, ok in (("small/layers", "small/out"), ("small/layers_unsorted", "small/out_unsorted")):
        layers = [int(l) for l in k[lk]]
        want = torch.from_numpy(k[ok])
        for f in range(centers.shape[0]):
            feat = RQAEFeature.from_quantizer(new, center=centers[f].numpy(), layers=list(layers))
            assert feat.num_quantizers == 64 and feat.dim == 4 and torch.equal(feat.layer_weights, lw)
            got = fo.intensity(sims, centers[f], codes, lw, layers)
            assert got.dtype == torch.float16 and got.shape == want[f].shape
            assert torch.equal(got, want[f]), (lk, f)


def test_reference_scripts3_get_activations_runs_on_new_class():
    """scripts/3_make_rqae_features.py:98-149 (FeatureHelper.get_activations) on the feature built from the new
    model class: same selected sequences in the same order and the same activation rows as the reference returned
    with its own model class, for two features, top_k 7 and 100, over three rounds of its 1024-sequence batching."""
    k = _load("kat_mining.npz")
    new = _new(0, dim=64, num_quantizers=64)
    assert np.array_equal(new.codebook.data[0].numpy(), k["cb0"])
    sims, lw = _reference_reads(new)
    assert torch.equal(lw, torch.from_numpy(k["lw"]))
    codes = torch.from_numpy(k["codes"].astype(np.int64))                  # (N, S, nq)
    S = codes.shape[1]
    layers = [int(l) for l in k["layers"]]
    for f in range(k["centers"].shape[0]):
        inten = fo.intensity(sims, torch.from_numpy(k["centers"][f]), codes, lw, layers)
        for top_k in (7, 100):
            got = fo.get_activations(inten.flatten(0, 1), layers, top_k, S)
            assert list(got.keys()) == layers
            for l in layers:
                seqs, acts = got[l]
                assert seqs == [int(s) for s in k[f"f{f}/k{top_k}/{l}/sequences"]], (f, top_k, l)
                want = k[f"f{f}/k{top_k}/{l}/activations"]
                assert acts.dtype == want.dtype and np.array_equal(acts.view(np.uint16), want.view(np.uint16)), (f, top_k, l)


def test_reference_server_tables_from_new_class():
    """demo/server/server.py:101-115 builds its engine table from subfeature_sims and layer_norms of the model:
    the new class's tables (5x5 Gram form, no (nq, K, D) intermediate) against the reference's own table."""
    from rqae_b200.search import engine_sims
    g = _load("kat_search.npz")
    for key, seed, kw in (("k81", 0, dict(dim=48, codebook_size=3, num_quantizers=160)),
                          ("k625", 1, dict(dim=32, num_quantizers=4))):
        new = _new(seed, **kw)
        ref = torch.from_numpy(g[f"{key}/sims"])
        K = new.codebook.shape[1]
        with torch.inference_mode():
            s_new = new.subfeature_sims
            got = engine_sims(new)
        assert s_new.shape == ref.shape == (kw["num_quantizers"], K, K) and s_new.dtype == got.dtype == torch.float16
        # a row's similarity with itself is 1, so the reference table's diagonal holds its layer norms in fp16
        assert torch.equal(new.layer_norms.half(), ref.diagonal(dim1=1, dim2=2).max(dim=-1).values), key
        # one fp16 ulp of a similarity (2^-11 at magnitude <= 1, the two forms sum in a different order), scaled by
        # the layer norm, plus the rounding of the scaled value
        assert float((got.float() - ref.float()).abs().max()) <= 2.0 ** -9 * float(new.layer_norms.max()), key
        assert float((got != ref).float().mean()) < 0.01, key
