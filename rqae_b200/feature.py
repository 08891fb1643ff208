"""``Feature`` / ``RQAEFeature`` -- host-side mirror of ``rqae/feature.py`` (harish-kamath/rqae) whose
``intensity`` runs on the B200 tensor cores (``rqae_intensity_f16`` in ``librqae_b200.so``).

Kept as in the reference: constructor arguments and attributes (feature.py:42-84), ``to_feature``
(:86-93), ``load_model`` (:95-100: fp16 layer weights = mean column norm of every out-projection),
``from_quantizer`` (:131-137), ``save`` / ``load`` (:139-153, plain ``np.savez``), and the signature
and result of ``intensity(token_indices, layers=None) -> (..., len(layers))`` fp16 (:102-129).

New: ``intensity_many`` evaluates MANY features over a code tensor in one launch sequence -- the inner
loop of ``scripts/3_make_rqae_features.py:98-114`` (one ``intensity`` call per feature and 1024-sequence
batch there) -- and returns the feature-major layout the mining step consumes.  ``precision="exact"``
(``rqae_intensity_exact_f16``) reproduces the reference's values bit for bit; the default ``"tc"`` GEMM
agrees with them within 2e-3.

There is no CPU path: code tensors must live on the GPU next to the model.
"""
from __future__ import annotations

import weakref
from typing import List, Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F

from . import _lib

TOKEN_TILE = 256   # the kernel writes whole tiles of 256 tokens


class Feature:
    """feature.py:9-40."""

    def __init__(self, id: str = "", explanation: str = "", scores: dict = {}, model: str = "", activations: list = []):
        self.id = str(id)
        self.explanation = str(explanation)
        self.scores = scores
        self.model = str(model)
        self.activations = activations  # list of {"text": [str], "activations": [float]}

    def save(self, file_path: str):
        np.savez(file_path, **self.__dict__)

    @classmethod
    def load(cls, file_path: str):
        params = dict(np.load(file_path, allow_pickle=True))
        for k, v in params.items():
            try:
                params[k] = v.item()
            except Exception:
                pass
        return cls(**params)


def layer_weights_f16(rqae) -> torch.Tensor:
    """feature.py:97-99, expression for expression (load-time host logic)."""
    return torch.tensor([l[1].weight.data.norm(dim=0).mean().item() for l in rqae.layers]).to(torch.float16)


def exact_sims(rqae, device) -> torch.Tensor:
    """The reference's own ``codebook_sims`` table (model.py:140-142, computed on the host as there) on ``device``, for
    ``precision="exact"``.  Cached per codebook storage and version; ``RQAE._apply`` drops the cache.  (The model's
    ``codebook_sims`` property of a CUDA model is a device matmul, which nothing shows to equal the host table.)"""
    cb = rqae.codebook
    key = (cb.untyped_storage().data_ptr(), cb._version, str(device))
    hit = rqae.__dict__.get("_exact_sims")
    if hit is None or hit[0] != key:
        n = F.normalize(cb.data.detach()[0].cpu().float(), dim=-1)
        hit = (key, (n @ n.T).half().to(device))
        rqae.__dict__["_exact_sims"] = hit
    return hit[1]


def _cuts(layers: Sequence[int]):
    cuts = sorted(set(int(l) for l in layers))
    pos = {l: i for i, l in enumerate(cuts)}
    return cuts, [pos[int(l)] for l in layers]


class IntensityWorkspace:
    """Caller-owned scratch of ``intensity_many``.  It keeps the tile-major copy of the code tensor between calls: a later
    call only rebuilds the feature operand (``rqae_intensity_again_f16``) when it passes the very tensor object of the
    previous call (held by a weak reference), unchanged since (same ``_version``, shape, strides and dtype), with the same
    cuts and codebook size, and ``intensity_many`` used that tensor as it is (int16 / int32 / int64 with rows of unit
    stride: no conversion, no ``.contiguous()`` copy).  A new tensor that happens to sit at a freed one's address, or a
    temporary copy of a tensor that was changed in place, never matches -- scripts/3_make_rqae_features.py:164-196 mines
    its features group by group over one code store."""

    def __init__(self):
        self.buf: Optional[torch.Tensor] = None
        self.key = None
        self.src: Optional[weakref.ref] = None   # the caller's code tensor behind ``key``


def intensity_many(rqae, token_indices: torch.Tensor, centers: torch.Tensor, layers: Sequence[int],
                   layer_weights: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                   workspace: Optional[IntensityWorkspace] = None, precision: str = "tc") -> torch.Tensor:
    """Intensities of F features over T tokens at the given layer cuts.

    token_indices (..., nq) integer codes on the GPU (int16 / int32 / int64); centers (F, nq) integer;
    returns fp16 (F, len(layers), T) with T = prod(...), feature-major: ``result[f, j]`` is the contiguous
    vector the reference calls ``all_intensities[:, j]`` for feature f (scripts/3:115-119).  ``out`` may be
    a caller-owned fp16 buffer (F, n_cuts_sorted, >= T rounded up to 256) to reuse between calls.

    precision="tc" (default): the tcgen05 GEMM, within 2e-3 of the reference, at most 64 distinct cuts.
    precision="exact": the reference's arithmetic bit for bit (rqae_intensity_exact_f16) for the given fp16 layer
    weights and codebook[0] -- note that ``layer_weights_f16`` computes the column norms on the model's device; any
    number of cuts; codes in [-K, 0) index as in the reference; ``out`` needs >= T rounded up to 8 columns; ``workspace``
    is not used."""
    if precision not in ("tc", "exact"):
        raise ValueError(f"unknown intensity precision {precision!r} (expected 'tc' or 'exact')")
    if rqae.quantization_method != "round_fsq":
        raise ValueError("Codebook sims only supported for round_fsq for now")   # model.py:139
    if not token_indices.is_cuda:
        raise RuntimeError("rqae_b200 intensity needs the code tensor on the GPU; there is no CPU fallback")
    dev = token_indices.device
    lib = _lib.load()
    codes = _lib.code_tensor(token_indices)
    nq_codes = codes.shape[-1]
    codes = codes.reshape(-1, nq_codes)
    if codes.stride(-1) != 1 or (codes.shape[0] > 1 and codes.stride(0) < nq_codes):
        codes = codes.contiguous()
    T = codes.shape[0]
    cuts, order = _cuts(layers)
    if cuts[0] < 0 or cuts[-1] >= min(nq_codes, centers.shape[-1]):
        raise IndexError(f"layer cut {cuts[-1]} outside the code tensors")
    centers = centers.to(device=dev, dtype=torch.int32).reshape(-1, centers.shape[-1]).contiguous()
    Fn = centers.shape[0]
    w = layer_weights if layer_weights is not None else layer_weights_f16(rqae)
    w = w.to(device=dev, dtype=torch.float16).contiguous()
    if w.numel() <= cuts[-1]:
        raise IndexError("layer_weights shorter than the deepest cut")
    cuts_arr = np.asarray(cuts, dtype=np.int32)
    pad = 8 if precision == "exact" else TOKEN_TILE
    T_pad = (T + pad - 1) // pad * pad
    if out is None:
        out = torch.empty(Fn, len(cuts), T_pad, dtype=torch.float16, device=dev)
    elif out.dtype != torch.float16 or out.device != dev or out.dim() != 3 or out.shape[0] != Fn \
            or out.shape[1] != len(cuts) or out.shape[2] < T_pad or not out.is_contiguous():
        raise RuntimeError(f"out must be a contiguous fp16 CUDA tensor (F, unique cuts, >= T rounded up to {pad})")
    if precision == "exact":
        if T > 0 and Fn > 0:
            sims = exact_sims(rqae, dev)
            with torch.cuda.device(dev):
                st = torch.cuda.current_stream(dev)
                rc = lib.rqae_intensity_exact_f16(
                    sims.data_ptr(), sims.shape[0], codes.data_ptr(), _lib.code_dtype(codes.dtype),
                    codes.stride(0) if T > 1 else nq_codes, T, centers.data_ptr(), centers.shape[1], Fn, w.data_ptr(),
                    cuts_arr.ctypes.data, len(cuts), out.data_ptr(), out.shape[2], st.cuda_stream)
            _lib.check(rc, "rqae_intensity_exact_f16")
            for t in (sims, w, centers, codes):
                t.record_stream(st)
    elif T > 0:
        cb_norm = F.normalize(rqae.codebook.data.detach()[0].to(device=dev, dtype=torch.float32), dim=-1).contiguous()
        K = cb_norm.shape[0]
        nbytes = lib.rqae_intensity_workspace_bytes(cuts_arr.ctypes.data, len(cuts), Fn, T)
        if nbytes == 0:
            raise NotImplementedError("unsupported intensity shape (at most 64 distinct cuts / 256 K-blocks)")
        # a copy made above is a new tensor on every call: its address and version say nothing about its contents
        own = codes.untyped_storage().data_ptr() == token_indices.untyped_storage().data_ptr()
        key = (codes.data_ptr(), token_indices._version, tuple(token_indices.shape), token_indices.stride(), codes.dtype,
               tuple(cuts), K, str(dev))
        ws, ws_ptr, ws_bytes = _lib.workspace(nbytes, dev, None if workspace is None else workspace.buf)
        # the codes of the previous call are still in the workspace only if it kept its buffer
        again = own and workspace is not None and workspace.key == key and workspace.src is not None \
            and workspace.src() is token_indices and ws is workspace.buf
        if workspace is not None and not again:
            workspace.buf, workspace.key = ws, None   # key set below, once the codes are in place
        with torch.cuda.device(dev):
            st = torch.cuda.current_stream(dev).cuda_stream
            if again:
                rc = lib.rqae_intensity_again_f16(cb_norm.data_ptr(), K, T, centers.data_ptr(), centers.shape[1], Fn, w.data_ptr(),
                                                  cuts_arr.ctypes.data, len(cuts), out.data_ptr(), out.shape[2], ws_ptr, ws_bytes, st)
            else:
                rc = lib.rqae_intensity_f16(
                    cb_norm.data_ptr(), K, codes.data_ptr(), _lib.code_dtype(codes.dtype),
                    codes.stride(0) if T > 1 else nq_codes, T, centers.data_ptr(), centers.shape[1], Fn, w.data_ptr(),
                    cuts_arr.ctypes.data, len(cuts), out.data_ptr(), out.shape[2], ws_ptr, ws_bytes, st)
        _lib.check(rc, "rqae_intensity_again_f16" if again else "rqae_intensity_f16")
        if workspace is not None:
            workspace.key, workspace.src = (key, weakref.ref(token_indices)) if own else (None, None)
        for t in (ws, cb_norm, w, centers, codes):
            t.record_stream(torch.cuda.current_stream(dev))
    res = out[:, :, :T]
    if order != list(range(len(cuts))):
        res = res[:, order]
    return res


def select_top_middle_bottom(intensities: torch.Tensor, top_k: int = 100, n: Optional[int] = None):
    """The selection of scripts/3_make_rqae_features.py:116-128 for every row of ``intensities`` (fp16, CUDA,
    (..., T) as returned by ``intensity_many``): positions of the ``top_k`` largest, the values around the
    median rank and the ``top_k`` smallest, without sorting the rows.  Returns (indices int32 (..., 3, top_k),
    values fp16 (..., 3, top_k)); order inside a window: value descending, then index ascending."""
    if not intensities.is_cuda or intensities.dtype != torch.float16:
        raise RuntimeError("select_top_middle_bottom needs an fp16 CUDA tensor; there is no CPU fallback")
    T = intensities.shape[-1] if n is None else int(n)
    v = intensities
    ok = v.dim() >= 1 and v.stride(-1) == 1 and v.data_ptr() % 16 == 0
    lead = v.shape[:-1]
    if ok and v.dim() > 1:
        rs = v.stride(-2)
        flat_ok = rs % 8 == 0 and rs >= (T + 7) // 8 * 8
        # all leading dims must collapse onto a single row stride
        exp = rs
        for d in range(v.dim() - 2, -1, -1):
            if v.shape[d] != 1 and v.stride(d) != exp:
                flat_ok = False
            exp *= v.shape[d]
        ok = flat_ok
    elif ok:
        rs = (T + 7) // 8 * 8
        ok = v.shape[0] >= rs or T % 8 == 0
    if not ok:   # repack into rows padded to a multiple of 8
        rs = (T + 7) // 8 * 8
        buf = torch.zeros(*lead, rs, dtype=torch.float16, device=v.device)
        buf[..., :T] = v[..., :T]
        v = buf
    rows = 1
    for d in lead:
        rows *= int(d)
    dev = v.device
    idx = torch.empty(*lead, 3, top_k, dtype=torch.int32, device=dev)
    val = torch.empty(*lead, 3, top_k, dtype=torch.float16, device=dev)
    if rows > 0:
        with torch.cuda.device(dev):
            rc = _lib.load().rqae_select_top_middle_bottom_f16(v.data_ptr(), rows, rs, T, int(top_k), idx.data_ptr(),
                                                                val.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(rc, "rqae_select_top_middle_bottom_f16")
        v.record_stream(torch.cuda.current_stream(dev))
    return idx, val


class RQAEFeature:
    """feature.py:42-153."""

    def __init__(self, id: str = "", explanations: List[str] = None, scores: List[dict] = None, activations: list = None,
                 model: str = "", num_quantizers: int = 1024, dim: int = 4, layers: List[int] = None,
                 layer_weights: List[float] = None, center: Optional[np.ndarray] = None, **kwargs):
        self.num_quantizers = num_quantizers
        self.dim = dim
        self.model = model
        self.id = id
        if layers is None:
            layers = [num_quantizers - 1]
        if layer_weights is None:
            layer_weights = np.ones(num_quantizers)
        if center is None:
            center = np.zeros((num_quantizers,))
        self.layers = layers
        self.layer_weights = torch.tensor(layer_weights)
        self.center = torch.tensor(center).int()
        if explanations is None:
            explanations = ["" for _ in layers]
        if scores is None:
            scores = [{} for _ in layers]
        if activations is None:
            activations = {k: [] for k in layers}
        self.explanations = explanations
        self.scores = scores
        self.activations = activations
        self.rqae = None

    def to_feature(self, layer: int = 0):
        return Feature(id=self.id, model=self.model, explanation=self.explanations[layer], scores=self.scores[layer],
                       activations=self.activations[self.layers[layer]])

    def load_model(self, rqae):
        self.rqae = rqae
        self.layer_weights = layer_weights_f16(rqae)
        return self

    def intensity(self, token_indices: torch.Tensor, layers=None, *, precision: str = "tc"):
        """feature.py:102-129: (..., num_quantizers) codes -> (..., len(layers)) fp16 intensities.  ``precision="exact"``
        gives the reference's values bit for bit, for any number of layers (``intensity_many``)."""
        if layers is None:
            layers = self.layers
        if self.rqae is None:
            raise ValueError("Model not loaded. Needed for intensity calculation.")
        res = intensity_many(self.rqae, token_indices, self.center.reshape(1, -1), layers, layer_weights=self.layer_weights,
                             precision=precision)
        return res[0].transpose(0, 1).reshape(*token_indices.shape[:-1], len(layers))

    @classmethod
    def from_quantizer(cls, quantizer, **kwargs):
        return cls(num_quantizers=quantizer.num_quantizers, dim=quantizer.codebook_dim, **kwargs).load_model(quantizer)

    def save(self, file_path: str):
        np.savez(file_path, **{k: v for k, v in self.__dict__.items() if k != "rqae"})

    @classmethod
    def load(cls, file_path: str):
        params = dict(np.load(file_path, allow_pickle=True))
        for k, v in params.items():
            try:
                if k == "explanations":
                    params[k] = [str(e) for e in v]
                params[k] = v.item()
            except Exception:
                pass
        return cls(**params)


def _sequences_in_order(picked: Sequence[int], seq_len: int) -> List[int]:
    """scripts/3:129-139: sequence numbers of the picked token positions, first appearance kept."""
    seen, out = set(), []
    for k in picked:
        s = int(k) // seq_len
        if s not in seen:
            seen.add(s)
            out.append(s)
    return out


def unique_token_indices(tokens: torch.Tensor) -> torch.Tensor:
    """scripts/3:53-82: for every distinct token id (ascending), the (sequence, position) of ONE occurrence chosen
    uniformly at random -- the first occurrence under a random permutation of all positions.  Draws exactly one
    ``torch.randperm(tokens.numel())`` from the global generator, as the reference does, so the same seed gives the same
    result.  Returns int32 (n_unique, 2)."""
    n, seq_len = tokens.numel(), tokens.shape[1]
    perm = torch.randperm(n)
    shuffled = tokens.flatten()[perm]
    uniq, inverse = torch.unique(shuffled, return_inverse=True)
    first = torch.full((uniq.numel(),), n, dtype=torch.int64).scatter_reduce(0, inverse, torch.arange(n), reduce="amin")
    where = perm[first]
    return torch.stack([where // seq_len, where % seq_len], dim=1).to(torch.int32)


class FeatureHelper:
    """``scripts/3_make_rqae_features.py:33-162`` without the Modal decorators: ``tokens`` (sequences, positions),
    ``texts`` (per sequence) and ``indices`` = the code store (sequences, positions, num_quantizers), here resident on
    the GPU.  ``get_activations`` keeps the reference's signature and result
    (``{layer: [{"text": ..., "activations": fp16 ndarray (positions,)}, ...]}``, sequences of the top / middle /
    bottom-k tokens in order of first appearance); ``get_activations_many`` does the same for a list of features with
    ONE intensity GEMM and ONE selection launch instead of one container per feature (scripts/3:189-191).  Equal
    intensities are ordered by token index (the reference's unstable argsort leaves them unspecified).  ``precision`` is
    that of ``intensity_many``: with ``"exact"`` every activation row equals the reference's bit for bit."""

    FEATURE_FOLDER = "/data/datasets/monology_pile/features/rqae-rqae-round_fsq-cbd4-cbs5-nq1024"   # scripts/3:152-158

    def __init__(self, tokens: torch.Tensor, texts: Sequence, indices: torch.Tensor, feature_folder: Optional[str] = None):
        if not indices.is_cuda:
            raise RuntimeError("FeatureHelper needs the code store on the GPU; there is no CPU fallback")
        if indices.dim() != 3 or tuple(indices.shape[:2]) != tuple(tokens.shape[:2]):
            raise ValueError("indices must be (sequences, positions, num_quantizers) matching tokens (sequences, positions)")
        self.tokens = tokens
        self.texts = texts
        self.indices = indices
        self.feature_folder = feature_folder or self.FEATURE_FOLDER

    def get_unique_token_indices(self):
        """scripts/3:53-82."""
        return unique_token_indices(self.tokens)

    def get_token_indices(self, index: torch.Tensor):
        """scripts/3:84-89."""
        if len(index.shape) == 1:
            return self.indices[index[0], index[1]]
        return self.indices[index[:, 0], index[:, 1]]

    def get_text(self, index: torch.Tensor):
        """scripts/3:91-96."""
        if index.shape[0] == 1:
            return self.texts[index[0].item()]
        return self.texts[index[0].item()][index[1].item()]

    def get_activations_many(self, features: Sequence["RQAEFeature"], layers: list = None, top_k: int = 100,
                             precision: str = "tc") -> List[dict]:
        if not features:
            return []
        if layers is None:
            layers = features[0].layers
        rqae = features[0].rqae
        if rqae is None:
            raise ValueError("Model not loaded. Needed for intensity calculation.")
        n_seq, seq_len = self.indices.shape[:2]
        centers = torch.stack([f.center.reshape(-1) for f in features])
        if "_workspace" not in self.__dict__:
            self._workspace = IntensityWorkspace()       # the code store's tile-major copy survives from one feature group to the next
        inten = intensity_many(rqae, self.indices, centers, layers, layer_weights=features[0].layer_weights,
                               workspace=self._workspace, precision=precision)                                 # (F, C, T)
        sel, _ = select_top_middle_bottom(inten, top_k)                                                        # (F, C, 3, k)
        sel = sel.cpu()
        mid = 2 * (top_k // 2)
        results = []
        for f in range(len(features)):
            activations = {}
            for j, l in enumerate(layers):
                picked = sel[f, j, 0].tolist() + sel[f, j, 1, :mid].tolist() + sel[f, j, 2].tolist()
                seqs = _sequences_in_order(picked, seq_len)
                rows = inten[f, j].reshape(n_seq, seq_len)[torch.tensor(seqs, device=inten.device)].cpu().numpy()
                activations[l] = [{"text": self.texts[s], "activations": rows[i]} for i, s in enumerate(seqs)]
            results.append(activations)
        return results

    def get_activations(self, rqae: "RQAEFeature", layers: list = None, top_k: int = 100, index=None,
                        precision: str = "tc"):
        """scripts/3:98-162."""
        import os
        activations = self.get_activations_many([rqae], layers=layers, top_k=top_k, precision=precision)[0]
        if index is not None:
            rqae.activations = activations
            os.makedirs(self.feature_folder, exist_ok=True)
            rqae.save(os.path.join(self.feature_folder, f"{index:06d}.npz"))
        return activations


SCRIPT3_LAYERS = [2, 4, 6, 8, 12, 16, 24, 32, 48, 64, 128, 256, 512, 1023]   # scripts/3:178


def make_feature(rqae, feature_helper: "FeatureHelper", num_tokens: int = 1024, layers: Optional[List[int]] = None,
                 top_k: int = 100, features_per_launch: int = 64, save: bool = True,
                 precision: str = "tc") -> List["RQAEFeature"]:
    """The driver of ``scripts/3_make_rqae_features.py:164-200`` on one GPU: one random occurrence per distinct token
    (``get_unique_token_indices``), the 200 lowest and highest token ids dropped, shuffled, the first ``num_tokens``
    kept (:167-172; two draws from the global generator, as in the reference); each becomes an ``RQAEFeature`` centred
    on that token's codes (:184-188) whose activations are mined over the whole store and saved as
    ``<feature_folder>/{i:06d}.npz`` (:150-158).  Where the reference spawns one container per feature (:189-191),
    ``features_per_launch`` features share one intensity GEMM and one selection launch (64 features x 14 cuts x
    4.7 M tokens of fp16 intensities = 8.4 GB).  ``precision="exact"`` mines from the reference's own intensity values."""
    import os
    layers = list(SCRIPT3_LAYERS if layers is None else layers)
    picks = feature_helper.get_unique_token_indices()
    picks = picks[200:-200]
    picks = picks[torch.randperm(picks.shape[0])]
    picks = picks[:num_tokens]
    centers = feature_helper.get_token_indices(picks)
    lw = layer_weights_f16(rqae)          # once: from_quantizer would recompute it (num_quantizers host syncs) per feature
    kw = {} if precision == "tc" else {"precision": precision}   # the default keeps get_activations_many's old call
    features = []
    for i in range(picks.shape[0]):
        f = RQAEFeature(num_quantizers=rqae.num_quantizers, dim=rqae.codebook_dim, center=centers[i].cpu().numpy(), layers=layers)
        f.rqae, f.layer_weights = rqae, lw
        features.append(f)
    for f0 in range(0, len(features), features_per_launch):
        group = features[f0:f0 + features_per_launch]
        for j, acts in enumerate(feature_helper.get_activations_many(group, layers=layers, top_k=top_k, **kw)):
            group[j].activations = acts
            if save:
                os.makedirs(feature_helper.feature_folder, exist_ok=True)
                group[j].save(os.path.join(feature_helper.feature_folder, f"{f0 + j:06d}.npz"))
    return features
