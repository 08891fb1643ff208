"""``RQAE`` -- host-side mirror of ``rqae.model.RQAE`` (harish-kamath/rqae, rqae/model.py) whose
hot path runs in the sm_100a kernels of ``librqae_b200.so``.

What is kept exactly as in the reference (so that ``rqae/llm.py`` hooks, ``rqae/feature.py`` and
``scripts/1_create_activations.py`` / ``scripts/3_make_rqae_features.py`` work unchanged):

* constructor signature and defaults, RNG consumption order of the random init (model.py:18-73);
* parameter / buffer names and shapes: ``layers.{l}.0.{weight,bias}``, ``layers.{l}.1.{weight,bias}``,
  ``codebook``, ``codebook_counts`` -- ``load_state_dict(strict=True)`` from the published
  safetensors works (model.py:89-96);
* ``forward(x, max_layers, temperature) -> (quantized_out fp32, indices int64)`` (model.py:199-230),
  ``decode`` / ``decode_from_codebook_values`` / ``indices_to_codebook_values`` (model.py:232-252),
  ``hook(**kwargs) -> hook_fn(module, input, output)`` (model.py:254-291), the derived tables
  ``codebook_sims / subfeatures / subfeature_sims / layer_norms`` (model.py:133-178).

What is new: ``encode(x, max_layers, out_dtype)`` (codes only), ``forward_host`` (host buffers in,
host buffers out, copies pipelined inside the C library).

The module holds no compute of its own: ``forward`` packs the weights once per weight version into
the streaming layout (``rqae_pack_weights``) and launches ONE fused kernel on the current CUDA stream
without synchronising.  CPU tensors are rejected -- there is deliberately no fallback path.
"""
from __future__ import annotations

import json
import math
import os
from typing import Callable, Optional, Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib

_FSQ = ("fsq", "round_fsq")


def _fsq_grid(codebook_size: int, codebook_dim: int, normalise: bool) -> torch.Tensor:
    """linspace(-1, 1, cbs)^cd, first coordinate slowest (itertools.product order), rows divided by
    their float64 norm for round_fsq with the zero row left untouched, then cast to fp32
    (model.py:63-72).  The axis is numpy's linspace, as in the reference (torch.linspace can differ from it
    in the last bit of a middle value, which changes a row of the normalised table).  sqrt and divide are correctly rounded in float64 both here and in numpy, so the table is
    bit-identical to the reference's (tests/test_model_host.py checks sizes 2..9)."""
    import numpy as np
    axis = torch.from_numpy(np.linspace(-1, 1, codebook_size))
    grid = torch.cartesian_prod(*([axis] * codebook_dim)).reshape(-1, codebook_dim)
    if normalise:
        n = grid.pow(2).sum(-1, keepdim=True).sqrt()
        grid = grid / torch.where(n == 0, torch.ones_like(n), n)
    return grid.to(torch.float32)


class RQAE(nn.Module):
    PRETRAINED = {
        "google/gemma-2-2b": "harish-kamath/rqae/gemma-2-2b",
        "rqae-rqae-round_fsq-cbd4-cbs5-nq1024": "harish-kamath/rqae/gemma-2-2b",
    }

    def __init__(self, dim: int = 2304, codebook_dim: int = 4, codebook_size: int = 5,
                 num_quantizers: int = 1024, quantization_method: str = "round_fsq", name: str = "", **kwargs):
        super().__init__()
        # Same module creation order as the reference so that torch.manual_seed(s); RQAE(...) yields the
        # same random weights (model.py:29-36): per layer Linear(dim, cd) then Linear(cd, dim).
        self.layers = nn.ModuleList(
            nn.ModuleList([nn.Linear(dim, codebook_dim), nn.Linear(codebook_dim, dim)])
            for _ in range(num_quantizers))
        rows = codebook_size ** codebook_dim if quantization_method in _FSQ else codebook_size
        self.codebook = nn.Parameter(torch.randn(num_quantizers, rows, codebook_dim))
        self.register_buffer("codebook_counts", torch.zeros(num_quantizers, rows), persistent=True)
        self.dim = dim
        self.quantization_method = quantization_method
        self.num_quantizers = num_quantizers
        self.codebook_dim = codebook_dim
        self.codebook_size = codebook_size
        self.name = name
        if quantization_method in _FSQ:
            with torch.no_grad():
                self.codebook.copy_(_fsq_grid(codebook_size, codebook_dim, quantization_method == "round_fsq"))
            self.codebook.requires_grad = False
        else:
            self.normalize_codebooks()
        self._packed = None          # (key, packed uint8 tensor, shared flag, search codebook tensor)
        self._static_weights = False

    # ------------------------------------------------------------------ loading (model.py:75-99)
    @classmethod
    def from_pretrained(cls, model_name: str):
        from huggingface_hub import hf_hub_download
        from safetensors import safe_open

        model_name = cls.PRETRAINED.get(model_name, model_name)
        username, reponame, *rest = model_name.split("/")
        folder = "/".join(rest)
        model_path = hf_hub_download(f"{username}/{reponame}", os.path.join(folder, "model.safetensors"))
        config_path = hf_hub_download(f"{username}/{reponame}", os.path.join(folder, "config.json"))
        with open(config_path, "r") as f:
            params = json.load(f)
        name = (f"rqae-{reponame}-{params['quantization_method']}-cbd{params['codebook_dim']}"
                f"-cbs{params['codebook_size']}-nq{params['num_quantizers']}")
        model = cls(**params, name=name)
        if model_path.endswith(".safetensors"):
            with safe_open(model_path, framework="pt") as f:
                state = {k: f.get_tensor(k) for k in f.keys()}
            model.load_state_dict(state, strict=True)
        elif model_path.endswith(".pt"):
            model.load_state_dict(torch.load(model_path, weights_only=True))
        else:
            raise ValueError(f"Unknown file extension for {model_path}")
        return model

    def update_codebook_counts(self, indices):
        """Codebook-usage EMA of the reference is disabled there (unconditional return, model.py:101-104)."""
        return

    def normalize_codebooks(self):
        """model.py:126-131: learned codebooks are re-normalised in place; fsq tables are left alone."""
        if self.quantization_method in _FSQ:
            return
        with torch.no_grad():
            self.codebook.copy_(self.codebook / self.codebook.norm(dim=-1, keepdim=True))

    # ------------------------------------------------------------------ packed weights
    def _apply(self, fn, *args, **kwargs):
        self._packed = None
        self.__dict__.pop("_tc_weights", None)
        for k in ("_codebook_sims", "_subfeatures", "_subfeature_sims", "_layer_norms", "_exact_sims"):
            self.__dict__.pop(k, None)
        return super()._apply(fn, *args, **kwargs)

    def load_state_dict(self, *args, **kwargs):
        self._packed = None
        return super().load_state_dict(*args, **kwargs)

    def repack(self):
        """Drop the packed copy of the weights (call after editing parameters through ``.data``)."""
        self._packed = None

    def freeze_packed(self, flag: bool = True):
        """Skip the per-call weight-version check (saves ~0.3 ms of Python per call when the weights
        are known not to change, e.g. inside an inference hook)."""
        self._static_weights = bool(flag)

    def _weights_key(self):
        w = self.layers[0][0].weight
        key = [w.device, w.data_ptr(), self.codebook.data_ptr()]
        if not self._static_weights:
            # learned codebooks are re-normalised in place by every forward (model.py:126-131): their version is
            # not part of the key, the per-layer tables are handed to the kernel separately (_learned_tables)
            learned = self.quantization_method not in _FSQ
            try:
                key.append(sum(p._version for p in self.parameters() if not (learned and p is self.codebook)))
            except RuntimeError:  # inference tensors carry no version counter
                pass
        return tuple(key)

    def _ensure_packed(self):
        key = self._weights_key()
        if self._packed is not None and self._packed[0] == key:
            return self._packed
        dev = self.layers[0][0].weight.device
        if dev.type != "cuda":
            raise RuntimeError("rqae_b200.RQAE computes on CUDA (sm_100a) only; move the module with .to('cuda'). "
                               "There is no CPU fallback.")
        if self.layers[0][0].weight.dtype != torch.float32:
            raise RuntimeError("rqae_b200.RQAE kernels are fp32 (the reference's compute dtype); call .float()")
        lib = _lib.load()
        nq, D, cd = self.num_quantizers, self.dim, self.codebook_dim
        K = self.codebook.shape[1]
        nbytes = lib.rqae_packed_bytes(nq, D, cd, K)
        if nbytes == 0:
            raise NotImplementedError(
                f"rqae_b200 kernels support codebook_dim == 4, dim <= 3584 and <= 65535 codebook rows "
                f"(got codebook_dim={cd}, dim={D}, rows={K})")
        with torch.no_grad():
            w_in = torch.stack([l[0].weight for l in self.layers]).contiguous()
            b_in = torch.stack([l[0].bias for l in self.layers]).contiguous()
            w_out = torch.stack([l[1].weight for l in self.layers]).contiguous()
            b_out = torch.stack([l[1].bias for l in self.layers]).contiguous()
            cb = self.codebook.detach()
            # The reference indexes codebook[layer] in forward; the single-table fast path is valid only
            # when every layer holds the same table (always true for fsq / round_fsq as constructed).
            shared = self.quantization_method in _FSQ and bool((cb == cb[:1]).all().item())
            cb_arg = cb[:1].contiguous() if shared else cb.contiguous()
            packed = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            stream = torch.cuda.current_stream(dev).cuda_stream
            with torch.cuda.device(dev):
                rc = lib.rqae_pack_weights(w_in.data_ptr(), b_in.data_ptr(), w_out.data_ptr(), b_out.data_ptr(),
                                           cb_arg.data_ptr(), int(shared), nq, D, cd, K, packed.data_ptr(), nbytes,
                                           stream)
            _lib.check(rc, "rqae_pack_weights")
            for t in (w_in, b_in, w_out, b_out):
                t.record_stream(torch.cuda.current_stream(dev))
        self._packed = (key, packed, shared, cb_arg)
        return self._packed

    # ------------------------------------------------------------------ hot path
    def _learned_tables(self, nq_run: int) -> torch.Tensor:
        """Reference quirk (model.py:126-131,196): ``quantize`` re-normalises the whole codebook parameter
        in place before EVERY layer, so layer l sees a table normalised l+1 times since the call began and
        the parameter ends up normalised nq_run times.  Reproduced here (iteration stops early once the
        normalisation reaches its fixed point) and the per-layer tables are handed to the kernel."""
        with torch.no_grad():
            cur = self.codebook.detach()
            tables = torch.empty_like(cur)
            done = 0
            for l in range(nq_run):
                nxt = cur / cur.norm(dim=-1, keepdim=True)
                tables[l] = nxt[l]
                done = l + 1
                fixed = bool((nxt == cur).all().item())
                cur = nxt
                if fixed:
                    break
            if done < nq_run:
                tables[done:nq_run] = cur[done:nq_run]
            if nq_run < tables.shape[0]:
                tables[nq_run:] = cur[nq_run:]
            self.codebook.copy_(cur)
        return tables.contiguous()

    def _run_forward(self, x: torch.Tensor, max_layers, temperature: float, want_q: bool, out_dtype: torch.dtype,
                     teacher: Optional[torch.Tensor] = None, want_z: bool = False):
        if self.training and temperature >= 1e-7:
            raise NotImplementedError("gumbel-softmax sampling (training with temperature >= 1e-7, model.py:180-185) "
                                      "is not part of the inference hot path")
        if not x.is_cuda:
            raise RuntimeError("rqae_b200.RQAE.forward needs a CUDA tensor; there is no CPU fallback")
        if x.dtype != torch.float32:
            raise RuntimeError(f"expected float32 activations (the reference hook calls .float() first), got {x.dtype}")
        if x.shape[-1] != self.dim:
            raise RuntimeError(f"last dimension must be {self.dim}, got {tuple(x.shape)}")
        nq_run = int(min(max_layers, self.num_quantizers))
        if nq_run <= 0:
            raise RuntimeError("max_layers must be >= 1 (the reference fails on an empty index list, model.py:226)")
        _, packed, shared, cb_arg = self._ensure_packed()
        if not shared and self.quantization_method not in _FSQ:
            cb_arg = self._learned_tables(nq_run)
        lib = _lib.load()
        xc = x.detach().contiguous()
        lead = xc.shape[:-1]
        n = xc.numel() // self.dim
        dev = xc.device
        codes = torch.empty(*lead, nq_run, dtype=out_dtype, device=dev)
        q = torch.empty_like(xc) if want_q else None
        z = torch.empty(*lead, nq_run, 4, dtype=torch.float32, device=dev) if want_z else None
        tch = None
        if teacher is not None:
            tch = teacher.to(device=dev, dtype=torch.int32).contiguous()
            assert tch.shape == codes.shape
        if n > 0:
            with torch.cuda.device(dev):
                rc = lib.rqae_forward_f32(
                    packed.data_ptr(), cb_arg.data_ptr(), int(shared), self.num_quantizers, nq_run, self.dim,
                    self.codebook_dim, self.codebook.shape[1], xc.data_ptr(), n, codes.data_ptr(),
                    _lib.code_dtype(out_dtype), nq_run,
                    0 if q is None else q.data_ptr(), 0 if tch is None else tch.data_ptr(),
                    0 if z is None else z.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
            _lib.check(rc, "rqae_forward_f32")
        return q, codes, z

    def forward(self, x, max_layers: int = float("inf"), temperature=0.0):
        """model.py:199-230.  Returns (quantized_out (B,S,D) fp32, indices (B,S,nq') int64)."""
        q, codes, _ = self._run_forward(x, max_layers, temperature, True, torch.int64)
        self.update_codebook_counts(codes)
        return q, codes

    def encode(self, x, max_layers: int = float("inf"), out_dtype: torch.dtype = torch.int64):
        """Codes only (forward without the reconstruction write).  ``out_dtype`` may be int16 / int32 / int64;
        every code is < codebook rows <= 65535."""
        if out_dtype == torch.int16 and self.codebook.shape[1] > 32768:
            raise ValueError(f"int16 cannot hold the codes of a {self.codebook.shape[1]}-row codebook; use int32")
        _, codes, _ = self._run_forward(x, max_layers, 0.0, False, out_dtype)
        return codes

    def indices_to_codebook_values(self, indices):
        """model.py:232-234 -- always the layer-0 table."""
        return self.codebook[0][indices]

    def _layer_mask(self, layers, nq_codes: int, dev):
        if layers is None:
            return None, nq_codes > 0
        mask = torch.zeros(max(nq_codes, 1), dtype=torch.uint8)
        any_sel = False
        for l in range(nq_codes):
            if l in layers:
                mask[l] = 1
                any_sel = True
        return mask.to(dev), any_sel

    def _run_decode(self, codes: Optional[torch.Tensor], cv: Optional[torch.Tensor], layers):
        src = codes if codes is not None else cv
        if not src.is_cuda:
            raise RuntimeError("rqae_b200.RQAE.decode needs CUDA tensors; there is no CPU fallback")
        _, packed, _, _ = self._ensure_packed()
        lib = _lib.load()
        dev = src.device
        if codes is not None:
            codes = _lib.code_tensor(codes).contiguous()
            lead, nq_codes = codes.shape[:-1], codes.shape[-1]
            code_dtype = _lib.code_dtype(codes.dtype)
        else:
            if cv.shape[-1] != self.codebook_dim:
                raise RuntimeError("codebook values must have last dimension codebook_dim")
            cv = cv.detach().to(torch.float32).contiguous()
            lead, nq_codes = cv.shape[:-2], cv.shape[-2]
            code_dtype = 0
        nq_codes = min(nq_codes, self.num_quantizers)
        mask, any_sel = self._layer_mask(layers, nq_codes, dev)
        if not any_sel:
            return None  # the reference returns its initial `quantized = None` (model.py:238,248)
        n = int(math.prod(lead)) if len(lead) else 1
        q = torch.empty(*lead, self.dim, dtype=torch.float32, device=dev)
        cb0 = self.codebook.detach()[0].contiguous()
        if n > 0:
            stride = (codes.shape[-1] if codes is not None else 0)
            if cv is not None and cv.shape[-2] != nq_codes:
                cv = cv[..., :nq_codes, :].contiguous()
            with torch.cuda.device(dev):
                rc = lib.rqae_decode_f32(
                    packed.data_ptr(), cb0.data_ptr(), self.num_quantizers, nq_codes, self.dim, self.codebook_dim,
                    self.codebook.shape[1], 0 if codes is None else codes.data_ptr(), code_dtype, stride,
                    0 if cv is None else cv.data_ptr(), 0 if mask is None else mask.data_ptr(), n, q.data_ptr(),
                    torch.cuda.current_stream(dev).cuda_stream)
            _lib.check(rc, "rqae_decode_f32")
        return q

    def decode_from_codebook_values(self, codebook_values, layers=None):
        """model.py:236-248."""
        return self._run_decode(None, codebook_values, layers)

    def decode(self, indices, layers=None, precision: str = "fp32"):
        """model.py:250-252: gather from codebook[0] + sum of the selected layers' out-projections, fused
        (the (B,S,nq,4) intermediate of the reference is never materialised).

        ``precision="fp32"`` (default) is bit-identical to the reference.  ``"f16"`` / ``"f16x3"`` opt in to the
        tensor-core path (one tcgen05 GEMM over the codes; fp16 operands, fp32 accumulation): relative error of
        the result about 2e-4 / 2e-5 (measured, max error over max |q|), 29x / 11x faster (1.0-1.15 PFLOP/s).  Not the default because it is not bit-exact."""
        if precision == "fp32":
            return self._run_decode(indices, None, layers)
        if precision not in ("f16", "f16x3"):
            raise ValueError("precision must be 'fp32', 'f16' or 'f16x3'")
        return self._run_decode_tc(indices, layers, 1 if precision == "f16" else 3)

    def _run_decode_tc(self, codes: torch.Tensor, layers, passes: int):
        if not codes.is_cuda:
            raise RuntimeError("rqae_b200.RQAE.decode needs CUDA tensors; there is no CPU fallback")
        lib = _lib.load()
        dev = codes.device
        codes = _lib.code_tensor(codes).contiguous()
        lead, nq_codes = codes.shape[:-1], min(codes.shape[-1], self.num_quantizers)
        mask, any_sel = self._layer_mask(layers, nq_codes, dev)
        if not any_sel:
            return None
        n = int(math.prod(lead)) if len(lead) else 1
        q = torch.empty(*lead, self.dim, dtype=torch.float32, device=dev)
        if n == 0:
            return q
        key = self._weights_key()
        cache = self.__dict__.get("_tc_weights")
        if cache is None or cache[0] != key:
            with torch.no_grad():
                w_out = torch.stack([l[1].weight.detach() for l in self.layers]).float().contiguous()   # (nq, D, 4)
                b_out = torch.stack([l[1].bias.detach() for l in self.layers]).float().contiguous()     # (nq, D)
            cache = (key, w_out, b_out)
            self.__dict__["_tc_weights"] = cache
        _, w_out, b_out = cache
        cb0 = self.codebook.detach()[0].float().contiguous()
        nbytes = lib.rqae_decode_tc_workspace_bytes(nq_codes, self.dim, n, passes)
        if nbytes == 0:
            raise NotImplementedError("tensor-core decode supports at most 3200 layer-passes (nq * passes)")
        ws, ws_ptr, ws_bytes = _lib.workspace(nbytes, dev)
        with torch.cuda.device(dev):
            rc = lib.rqae_decode_tc_f32(
                w_out.data_ptr(), b_out.data_ptr(), cb0.data_ptr(), self.num_quantizers, nq_codes, self.dim,
                self.codebook_dim, self.codebook.shape[1], codes.data_ptr(), _lib.code_dtype(codes.dtype),
                codes.shape[-1], 0 if mask is None else mask.data_ptr(), n, q.data_ptr(), passes, ws_ptr, ws_bytes,
                torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(rc, "rqae_decode_tc_f32")
        for t in (ws, cb0, codes):
            t.record_stream(torch.cuda.current_stream(dev))
        return q

    def forward_host(self, x_host: torch.Tensor, max_layers=float("inf"), want_q: bool = True,
                     out_dtype: torch.dtype = torch.int64, chunk_tokens: int = 9472, device=None,
                     out: Optional[tuple] = None, code_transfer: Optional[str] = None,
                     widen_threads: Optional[int] = None):
        """End-to-end variant for host-resident activations: ``x_host`` is a CPU tensor (pinned for full
        copy speed); codes and reconstruction come back in (pinned) CPU tensors.  H2D copy, kernel and D2H
        copies of consecutive chunks overlap inside ``rqae_forward_host_f32``.  ``out=(q, codes)`` reuses
        caller-owned (pinned) result tensors -- page-locking fresh result buffers costs more than the whole
        computation, so a caller that loops should allocate them once.  The default chunk is 4 full waves of
        the forward kernel (148 SMs x 16 tokens): the first H2D and the last D2H, which nothing overlaps, are
        1 % of a 1 Mi-token call.  ``code_transfer`` = "direct" | "narrow" | "auto" and ``widen_threads`` set the
        process-wide pipeline options of ``rqae_forward_host_config`` (see include/rqae_b200.h)."""
        if code_transfer is not None or widen_threads is not None:
            mode = {None: -1, "auto": 0, "narrow": 1, "direct": 2}[code_transfer]
            _lib.check(_lib.load().rqae_forward_host_config(mode, -1 if widen_threads is None else int(widen_threads)),
                       "rqae_forward_host_config")
        if x_host.is_cuda or x_host.dtype != torch.float32:
            raise RuntimeError("forward_host expects a float32 CPU tensor")
        if x_host.shape[-1] != self.dim:
            raise RuntimeError(f"last dimension must be {self.dim}, got {tuple(x_host.shape)}")
        nq_run = int(min(max_layers, self.num_quantizers))
        if nq_run <= 0:
            raise RuntimeError("max_layers must be >= 1")
        _, packed, shared, cb_arg = self._ensure_packed()
        if not shared and self.quantization_method not in _FSQ:
            cb_arg = self._learned_tables(nq_run)
        dev = packed.device
        xc = x_host.contiguous()
        lead = xc.shape[:-1]
        n = xc.numel() // self.dim
        pin = torch.cuda.is_available()
        if out is not None:
            q, codes = out
            if codes is None or codes.is_cuda or codes.dtype != out_dtype or tuple(codes.shape) != (*lead, nq_run) \
                    or not codes.is_contiguous():
                raise RuntimeError("out[1] must be a contiguous CPU tensor of shape (*lead, nq') and dtype out_dtype")
            if want_q and (q is None or q.is_cuda or q.dtype != torch.float32 or tuple(q.shape) != (*lead, self.dim)
                           or not q.is_contiguous()):
                raise RuntimeError("out[0] must be a contiguous float32 CPU tensor shaped like x_host")
            if not want_q:
                q = None
        else:
            codes = torch.empty(*lead, nq_run, dtype=out_dtype, pin_memory=pin)
            q = torch.empty(*lead, self.dim, dtype=torch.float32, pin_memory=pin) if want_q else None
        torch.cuda.current_stream(dev).synchronize()  # packed weights are produced on the current stream
        if n > 0:
            with torch.cuda.device(dev):
                rc = _lib.load().rqae_forward_host_f32(
                    packed.data_ptr(), cb_arg.data_ptr(), int(shared), self.num_quantizers, nq_run, self.dim,
                    self.codebook_dim, self.codebook.shape[1], xc.data_ptr(), n, codes.data_ptr(),
                    _lib.code_dtype(out_dtype), 0 if q is None else q.data_ptr(), int(chunk_tokens))
            _lib.check(rc, "rqae_forward_host_f32")
        return q, codes

    # ------------------------------------------------------------------ hook (model.py:254-291)
    @staticmethod
    def _gemma_rmsnorm(llm):
        """The final RMSNorm of the reference's Gemma-2 adapter (rqae/llm.py:60-73: ``norm`` = ``model.model.norm``,
        ``denorm`` divides by ``1 + norm.weight`` and by ``rsqrt(mean(hs^2) + 1e-6)``), when ``llm`` is that adapter:
        (weight, eps) or None.  Only the (1 + w) RMSNorm of the Gemma family qualifies for the fused hook."""
        try:
            norm = llm.model.model.norm
        except AttributeError:
            return None
        if "Gemma" not in type(norm).__name__ or not hasattr(norm, "weight") or not hasattr(norm, "eps"):
            return None
        if type(llm).__name__ != "Gemma2":         # another adapter may define norm / denorm differently
            return None
        return norm.weight, float(norm.eps)

    def hook_rmsnorm_(self, hidden: torch.Tensor, rms_weight: torch.Tensor, rms_eps: float = 1e-6, skip_bos: bool = True,
                      replace: bool = True, return_codes: bool = False, out_dtype: torch.dtype = torch.int64):
        """The body of ``hook_fn`` (model.py:276-289) for the Gemma-2 RMSNorm (llm.py:65-73) as ONE kernel launch on the
        current stream (``rqae_hook_rmsnorm``): ``hidden`` (B, S, dim) fp16 / bf16 / fp32, contiguous, is normalised on
        the way into the layer loop and -- when ``replace`` -- overwritten in place with the de-normalised
        reconstruction (position 0 of every sequence untouched when ``skip_bos``).  Returns the codes (B, S, nq) when
        ``return_codes``, else None."""
        hd = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}.get(hidden.dtype)
        if hd is None or not hidden.is_cuda or hidden.dim() != 3 or hidden.shape[-1] != self.dim or not hidden.is_contiguous():
            raise RuntimeError("hook_rmsnorm_ needs a contiguous CUDA tensor (B, S, dim) of fp16 / bf16 / fp32")
        if self.training:
            raise NotImplementedError("the fused hook is an inference path (eval mode)")
        _, packed, shared, cb_arg = self._ensure_packed()
        if not shared or self.quantization_method not in _FSQ:
            raise NotImplementedError("the fused hook supports the shared fsq / round_fsq codebook")
        dev = hidden.device
        cache = self.__dict__.get("_rms_w")
        if cache is None or cache[0] is not rms_weight or cache[1].device != dev or cache[2] != rms_weight._version:
            cache = (rms_weight, rms_weight.detach().to(device=dev, dtype=torch.float32).contiguous(), rms_weight._version)
            self.__dict__["_rms_w"] = cache
        w = cache[1]
        if w.numel() != self.dim:
            raise RuntimeError(f"rms_weight must have {self.dim} elements")
        B, S, _ = hidden.shape
        n = B * S
        codes = torch.empty(B, S, self.num_quantizers, dtype=out_dtype, device=dev) if return_codes else None
        if n > 0:
            with torch.cuda.device(dev):
                rc = _lib.load().rqae_hook_rmsnorm(
                    packed.data_ptr(), cb_arg.data_ptr(), int(shared), self.num_quantizers, self.num_quantizers, self.dim,
                    self.codebook_dim, self.codebook.shape[1], hidden.data_ptr(), hd, n, S, w.data_ptr(), float(rms_eps),
                    int(bool(skip_bos)), int(bool(replace)), 0 if codes is None else codes.data_ptr(),
                    _lib.code_dtype(out_dtype), self.num_quantizers,
                    torch.cuda.current_stream(dev).cuda_stream)
            _lib.check(rc, "rqae_hook_rmsnorm")
        return codes

    def hook(self, **kwargs) -> Callable:
        """model.py:254-291.  Same kwargs (``llm=`` or ``norm=`` / ``denorm=``, ``store``, ``skip_bos``, ``replace``).

        Fused fast path (SURVEY 8f-2): when the norm is the Gemma-2 RMSNorm -- ``llm`` is the reference's ``Gemma2``
        adapter, or ``rms_weight=`` / ``rms_eps=`` are passed -- and no ``store`` consumer is given, the whole body of
        ``hook_fn`` (float cast, norm, forward, denorm, BOS passthrough, cast back, in-place replace) is ONE kernel
        launch (``rqae_hook_rmsnorm``) on the current stream.  ``fused=False`` forces the generic path."""
        if "llm" in kwargs:
            llm = kwargs.pop("llm")
            assert hasattr(llm, "norm") and hasattr(llm, "denorm"), "RQAE hook requires norm and denorm from LLM"
            if "rms_weight" not in kwargs:
                g = self._gemma_rmsnorm(llm)
                if g is not None:
                    kwargs["rms_weight"], kwargs["rms_eps"] = g
            return self.hook(norm=llm.norm, denorm=llm.denorm, **kwargs)
        user_store = kwargs.get("store")
        if user_store is None:
            # the reference clones five full tensors per call even for its default no-op store (model.py:258,278-288);
            # without a consumer the clones are skipped (SURVEY 8f-2: "zero clones when store is the default no-op")
            def store(name, value):
                return None
        else:
            def store(name, value):
                return user_store(name, value.detach().clone())
        skip_bos = kwargs.get("skip_bos", True)
        replace = kwargs.get("replace", True)
        if "norm" not in kwargs:
            raise ValueError("RQAE hook requires norm from LLM")
        if "denorm" not in kwargs:
            raise ValueError("RQAE hook requires denorm from LLM")
        norm, denorm = kwargs["norm"], kwargs["denorm"]
        rms_weight = kwargs.get("rms_weight")
        rms_eps = float(kwargs.get("rms_eps", 1e-6))
        want_fused = kwargs.get("fused", True) and user_store is None and rms_weight is not None

        def hook_fused(out0) -> bool:
            """One launch for the whole hook body; False when this call does not qualify."""
            if out0.dtype not in (torch.float32, torch.float16, torch.bfloat16) or not out0.is_cuda or out0.dim() != 3 \
                    or out0.shape[-1] != self.dim or not out0.is_contiguous():
                return False
            if self.training or self.quantization_method not in _FSQ or not self._ensure_packed()[2]:
                return False
            self.hook_rmsnorm_(out0, rms_weight, rms_eps, skip_bos=skip_bos, replace=replace)
            return True

        def hook_fn(module, input, output):
            if want_fused and hook_fused(output[0].data):
                return
            hs = output[0].float()                      # (B, S, dim)
            store("original", hs)
            rms_hs = norm(hs)
            store("normed", rms_hs)
            q_out, indices = self(rms_hs)               # one fused kernel on the current stream, no sync
            store("quantized", q_out)
            store("indices", indices)
            q_out = denorm(q_out, hs)
            if skip_bos:
                q_out[:, 0] = hs[:, 0]
            store("new", q_out)
            if replace:
                output[0].data.copy_(q_out)

        return hook_fn

    # ------------------------------------------------------------------ derived tables (model.py:133-178)
    @property
    def codebook_sims(self):
        if "_codebook_sims" not in self.__dict__:
            if self.quantization_method != "round_fsq":
                raise ValueError("Codebook sims only supported for round_fsq for now")
            cb = F.normalize(self.codebook.data.detach().clone()[0], dim=-1)
            self.__dict__["_codebook_sims"] = (cb @ cb.T).to(torch.float16)
        return self.__dict__["_codebook_sims"]

    @property
    def subfeatures(self):
        if "_subfeatures" not in self.__dict__:
            self.__dict__["_subfeatures"] = torch.stack(
                [self.layers[l][1](self.codebook[l]) for l in range(self.num_quantizers)])
        return self.__dict__["_subfeatures"]  # (num_quantizers, rows, dim)

    @property
    def subfeature_sims(self):
        """model.py:157-167: cosine similarities of the rows of ``subfeatures`` per layer, fp16 (nq, K, K).
        The reference materialises ``subfeatures`` (nq, K, D) fp32 -- 5.9 GB at the 2B shape -- to get them.
        A subfeature is the affine image ``W_out[l] c + b_out[l]``, so all K*K inner products of a layer follow
        from the 5x5 Gram matrix of ``[W_out[l] | b_out[l]]`` (SURVEY 8f-4): ``<s_a, s_b> = [c_a;1]^T M_l [c_b;1]``.
        Same values up to fp32 rounding of a different summation order (a few fp16 ulps in rare entries)."""
        if "_subfeature_sims" not in self.__dict__:
            with torch.no_grad():
                w = torch.stack([l[1].weight.detach() for l in self.layers]).float()          # (nq, D, cd)
                b = torch.stack([l[1].bias.detach() for l in self.layers]).float()            # (nq, D)
                a = torch.cat([w, b.unsqueeze(-1)], dim=-1)                                   # (nq, D, cd+1)
                m = a.transpose(1, 2) @ a                                                      # (nq, cd+1, cd+1)
                cb = self.codebook.detach().float()                                            # (nq, K, cd)
                x = torch.cat([cb, torch.ones_like(cb[..., :1])], dim=-1)                      # (nq, K, cd+1)
                out = torch.empty(cb.shape[0], cb.shape[1], cb.shape[1], dtype=torch.float16, device=cb.device)
                step = 64
                for l0 in range(0, cb.shape[0], step):
                    xs, ms = x[l0:l0 + step], m[l0:l0 + step]
                    g = xs @ ms @ xs.transpose(1, 2)                                           # (s, K, K) inner products
                    n = g.diagonal(dim1=1, dim2=2).clamp_min(0).sqrt().clamp_min(1e-12)         # F.normalize eps
                    out[l0:l0 + step] = (g / (n.unsqueeze(2) * n.unsqueeze(1))).to(torch.float16)
            self.__dict__["_subfeature_sims"] = out
        return self.__dict__["_subfeature_sims"]

    @property
    def layer_norms(self):
        if "_layer_norms" not in self.__dict__:
            self.__dict__["_layer_norms"] = torch.tensor(
                [l[1].weight.data.norm(dim=0).mean().item() for l in self.layers],
                device=self.layers[0][1].weight.device)
        return self.__dict__["_layer_norms"]
