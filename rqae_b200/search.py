"""``IntensityEngine`` -- host-side mirror of the nearest-example search of the reference's demo server
(harish-kamath/rqae, ``demo/server/server.py:71-325``) without the Modal plumbing (SURVEY 8f-3).

Kept as in the reference: what ``setup()`` leaves on the object (``sims`` = ``subfeature_sims * layer_norms`` in
fp16, server.py:104-115; ``activations`` = the code store with the BOS position dropped, :118-139) and
``find_examples(idx=None, activation=None, top_examples=30, middle_examples=10, bottom_examples=10, layers=[...])``
as a generator that yields, after every layer of ``layers``, ``({"top"|"middle"|"bottom": {"indices": int32
(Sq, k) CPU, "intensities": fp16 (Sq, k, S) CPU}}, layer)`` (:159-325), with the same ``ValueError`` for a missing
or doubled query (:174-182).

Different by design: the code store is ONE resident CUDA tensor (N, S, nq) instead of a Python list of CPU
shards copied to the GPU range by range (a B200 holds the whole 36 864 x 127 x 1024 store: 9.6 GB as int16); the
gather + sum + accumulate of :204-263 is one kernel per layer range (``rqae_search_accumulate_f16``) that never
materialises the (1024, 127, 127, 64) gathered tensor; the ``argsort`` over sequences of :268 is the exact radix
select of the mining path (``rqae_select_top_middle_bottom_f16``).  Order among equal maxima: value descending,
sequence index ascending (the reference's unstable ``argsort`` leaves it unspecified).

There is no CPU path: model and code store must be on the GPU.
"""
from __future__ import annotations

from typing import Iterator, List, Optional, Sequence, Tuple, Union

import torch

from . import _lib, store

SQ_PAD = 128          # rq_search.cuh SR_Q: query positions are padded to one 256-byte row
SELECT_KMAX = 256     # rq_mine.cuh MN_KMAX
SERVER_LAYERS = [4, 6, 8, 12, 16, 24, 32, 48, 64, 128, 256, 512, 1023]   # server.py:167


def engine_sims(model, mode: str = "projected") -> torch.Tensor:
    """server.py:103-115: the (nq, K, K) fp16 table of the engine."""
    if mode == "original":
        sims = model.codebook_sims.unsqueeze(0).repeat(model.num_quantizers, 1, 1)
    elif mode == "projected":
        sims = model.subfeature_sims.clone()
    else:
        raise ValueError(f"Invalid mode: {mode}")
    sims *= model.layer_norms.to(sims.device).unsqueeze(-1).unsqueeze(-1)
    return sims.detach().contiguous()


TC_ROWS = 640         # rq_intensity.cuh IT_LUT_ROWS: rows per layer of the factor tables (codebook rows + the zero row)


def rank_factors(model, mode: str = "projected") -> torch.Tensor:
    """Unit vectors f_l(c), (nq, K, R) float64, with  table_mode[l][a][b] = f_l(a) . f_l(b)  before the fp16 rounding and
    the layer norm of server.py:104-115.  "projected" (rqae/model.py:145-167): a subfeature is the affine image
    W_out[l] c + b_out[l], so its cosine with another one is that of R_l [c; 1] with R_l^T R_l the 5x5 Gram matrix of
    [W_out[l] | b_out[l]] (R = 5).  "original" (model.py:140-142): the normalised codebook rows themselves (R = 4)."""
    with torch.no_grad():
        cb = model.codebook.detach().double()                                                # (nq or 1, K, cd)
        if mode == "original":
            f = torch.nn.functional.normalize(cb[0], dim=-1)
            return f.unsqueeze(0).repeat(model.num_quantizers, 1, 1)
        if mode != "projected":
            raise ValueError(f"Invalid mode: {mode}")
        w = torch.stack([l[1].weight.detach() for l in model.layers]).double()              # (nq, D, cd)
        b = torch.stack([l[1].bias.detach() for l in model.layers]).double()                # (nq, D)
        g = torch.cat([w, b.unsqueeze(-1)], dim=-1)
        m = g.transpose(1, 2) @ g                                                            # (nq, cd+1, cd+1)
        evals, evecs = torch.linalg.eigh(m)
        r = evals.clamp_min(0).sqrt().unsqueeze(-1) * evecs.transpose(1, 2)                  # R^T R = M
        if cb.shape[0] == 1:
            cb = cb.expand(w.shape[0], -1, -1)
        x = torch.cat([cb, torch.ones_like(cb[..., :1])], dim=-1)
        u = x @ r.transpose(1, 2)
        n = u.norm(dim=-1, keepdim=True)
        return torch.where(n > 1e-12, u / n.clamp_min(1e-12), torch.zeros_like(u))


class IntensityEngine:
    """server.py:71-325.  ``activations``: (N, S, nq) integer CUDA tensor, or a list of such shards (they are
    concatenated once; the reference keeps the list).  ``sims``: the fp16 table, or ``model`` to build it.

    ``precision="tc"`` (opt-in, needs ``model``): the per-position maxima that RANK the sequences come from the
    tensor-core form of the accumulation (``rqae_search_tc_maxima_f16``: the table is rank 5 per layer, fp16 factors,
    fp32 running prefix, no per-chunk roundings) -- a few fp16 steps from the reference's values, so sequences whose
    maxima are that close to a window boundary can swap; the ``intensities`` reported for the selected sequences are
    recomputed with the reference's exact arithmetic (``rqae_search_rows_f16``).  Default ``"exact"``."""

    def __init__(self, model=None, activations: Union[torch.Tensor, Sequence[torch.Tensor], None] = None, *,
                 sims: Optional[torch.Tensor] = None, mode: str = "projected", dataset: str = "monology_pile",
                 model_id: str = "rqae-rqae-round_fsq-cbd4-cbs5-nq1024", precision: str = "exact"):
        self.dataset = dataset
        self.model_id = model_id
        if precision not in ("exact", "tc"):
            raise ValueError(f"precision must be 'exact' or 'tc', got {precision!r}")
        if precision == "tc" and model is None:
            raise ValueError("precision='tc' builds its factor tables from the model: pass model")
        self.precision = precision
        if sims is None:
            if model is None:
                raise ValueError("Must specify either model or sims")
            sims = engine_sims(model, mode)
        if not sims.is_cuda:
            raise RuntimeError("IntensityEngine needs CUDA tensors; there is no CPU fallback")
        if sims.dim() != 3 or sims.shape[1] != sims.shape[2]:
            raise ValueError(f"sims must be (num_quantizers, K, K), got {tuple(sims.shape)}")
        self.sims = sims.to(torch.float16).contiguous()
        if activations is None:
            raise ValueError("Must specify activations")
        if not isinstance(activations, torch.Tensor):
            activations = torch.cat([a.to(self.sims.device) for a in activations], dim=0)
        if not activations.is_cuda:
            raise RuntimeError("IntensityEngine needs the code store on the GPU; there is no CPU fallback")
        if activations.dim() != 3 or _lib.code_dtype(activations.dtype) is None:
            raise ValueError("activations must be an int16/int32/int64 tensor (sequences, positions, num_quantizers)")
        if activations.shape[0] == 0 or activations.shape[1] == 0:
            raise ValueError("the code store is empty")
        self.activations = activations.contiguous()
        if precision == "tc":
            self._setup_tc(model, mode)

    def _setup_tc(self, model, mode: str) -> None:
        """Factor tables (fp16, 8 values per row, layers padded to a multiple of 8) and the 8-layer block-major copy of
        the code store that the GEMM streams; once per engine."""
        dev = self.sims.device
        N, S, nq_codes = self.activations.shape
        nq, K = self.sims.shape[0], self.sims.shape[1]
        if S > 128 or K + 1 > TC_ROWS:
            raise NotImplementedError("precision='tc': at most 128 positions per sequence and 639 codebook rows")
        f = rank_factors(model, mode).to(dev)                                                 # (nq, K, R) float64
        norms = model.layer_norms.to(dev).double().reshape(-1, 1, 1)
        lp = (nq + 7) // 8 * 8
        self._vtab = torch.zeros(lp, TC_ROWS, 8, dtype=torch.float16, device=dev)
        self._utab = torch.zeros(lp, TC_ROWS, 8, dtype=torch.float16, device=dev)
        self._vtab[:nq, :K, :f.shape[-1]] = f.to(torch.float16)
        self._utab[:nq, :K, :f.shape[-1]] = (f * norms).to(torch.float16)
        lib = _lib.load()
        nbytes = lib.rqae_search_tc_store_bytes(N, nq_codes)
        self._store_tc = torch.empty(nbytes // 2, dtype=torch.int16, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.rqae_search_tc_pack_store(self.activations.data_ptr(), _lib.code_dtype(self.activations.dtype), nq_codes,
                                                    N, S, nq_codes, K, self._store_tc.data_ptr(), nbytes,
                                                    torch.cuda.current_stream(dev).cuda_stream), "rqae_search_tc_pack_store")

    def maxima_tc(self, query: torch.Tensor, layers: Sequence[int], padded: bool = False) -> torch.Tensor:
        """(len(layers), Sq, N) fp16: max over the positions of every sequence of the running accumulation after each
        range of ``layers`` -- ``max_values.T`` of server.py:267 for all cuts, from ONE tensor-core launch (a view of
        a buffer whose rows are padded: what ``select_top_middle_bottom`` ranks)."""
        if self.precision != "tc":
            raise RuntimeError("maxima_tc needs an engine built with precision='tc'")
        layers = [int(l) for l in layers]
        if not layers or any(b <= a for a, b in zip([0] + layers[:-1], layers)):
            raise ValueError("layers must be strictly ascending positive layer indices")
        N, S, nq_codes = self.activations.shape
        nq, K = self.sims.shape[0], self.sims.shape[1]
        if layers[-1] > nq or layers[-1] > nq_codes:
            raise ValueError(f"max(layers)={layers[-1]} exceeds the {min(nq, nq_codes)} layers of the table / code store")
        dev = self.sims.device
        Sq = query.shape[0]
        lib = _lib.load()
        lh = torch.tensor(layers, dtype=torch.int32)
        wbytes = lib.rqae_search_tc_workspace_bytes(lh.data_ptr(), len(layers))
        if wbytes == 0:
            raise NotImplementedError("precision='tc': too many layer ranges for one launch")
        ws, ws_ptr, ws_bytes = _lib.workspace(wbytes, dev)
        stride = ((N + 1) // 2 * 2 + 7) // 8 * 8
        out = torch.empty(len(layers), SQ_PAD, stride, dtype=torch.float16, device=dev)
        if stride > (N + 1) // 2 * 2:     # the kernel writes two columns per unit; the selection's 16-byte loads touch the padding
            out[:, :, (N + 1) // 2 * 2:].zero_()
        with torch.cuda.device(dev):
            st = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(lib.rqae_search_tc_maxima_f16(self._store_tc.data_ptr(), N, S, nq_codes, self._vtab.data_ptr(),
                                                    self._utab.data_ptr(), self._vtab.shape[0], K, query.data_ptr(),
                                                    query.stride(0), Sq, lh.data_ptr(), len(layers), out.data_ptr(), stride,
                                                    ws_ptr, ws_bytes, st), "rqae_search_tc_maxima_f16")
        ws.record_stream(torch.cuda.current_stream(dev))
        return out[:, :, :N] if padded else out[:, :Sq, :N]     # padded: all 128 rows per cut (rows >= Sq are zero)

    def rows_exact(self, table: torch.Tensor, sel: torch.Tensor, layers: Sequence[int], first_range: Optional[int] = None) -> torch.Tensor:
        """``intensity_accumulation[sel[..., q, j], :, q]`` (server.py:290-305) recomputed with the reference's arithmetic
        for the selected sequences only.  ``table``: the query's rows of the engine table as they lie (``_build_qrows``).
        ``sel`` (Sq, n_sel): after all ranges of ``layers`` -> (Sq, n_sel, S) fp16.  ``sel`` (C, Sq, n_sel) with
        ``first_range``: selection c after the ranges 0 .. first_range + c -> (C, Sq, n_sel, S), one launch."""
        N, S, nq_codes = self.activations.shape
        K = self.sims.shape[1]
        dev = self.sims.device
        sel = sel.to(torch.int32).contiguous()
        single = sel.dim() == 2
        if single:
            sel = sel.unsqueeze(0)
            first_range = len(layers) - 1
        C, Sq, n_sel = sel.shape
        out = torch.empty(C, Sq, n_sel, S, dtype=torch.float16, device=dev)
        lh = torch.tensor([int(l) for l in layers], dtype=torch.int32)
        with torch.cuda.device(dev):
            _lib.check(_lib.load().rqae_search_rows_f16(table.data_ptr(), K, self.activations.data_ptr(),
                                                       _lib.code_dtype(self.activations.dtype), nq_codes, N, S, sel.data_ptr(), Sq,
                                                       n_sel, lh.data_ptr(), int(first_range), C, out.data_ptr(),
                                                       torch.cuda.current_stream(dev).cuda_stream), "rqae_search_rows_f16")
        return out[0] if single else out

    def _pinned(self, name: str, shape, dtype) -> torch.Tensor:
        cache = self.__dict__.setdefault("_pinned_cache", {})
        t = cache.get(name)
        n = 1
        for d in shape:
            n *= int(d)
        if t is None or t.dtype != dtype or t.numel() < n:
            t = torch.empty(n, dtype=dtype, pin_memory=True)
            cache[name] = t
        return t[:n].view(*shape)

    def _build_qrows(self, query: torch.Tensor, L: int) -> torch.Tensor:
        """server.py:183-196: ``query_sims[l, q] = sims[l, query[q, l]]`` as one (L, Sq, K) fp16 tensor -- what ``rows_exact`` gathers from."""
        lib = _lib.load()
        K = self.sims.shape[1]
        dev = self.sims.device
        Sq = query.shape[0]
        out = torch.empty(L, Sq, K, dtype=torch.float16, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.rqae_search_build_qrows_f16(self.sims.data_ptr(), K, query.data_ptr(), query.stride(0), Sq, L,
                                                      out.data_ptr(), out.numel() * 2, torch.cuda.current_stream(dev).cuda_stream),
                       "rqae_search_build_qrows_f16")
        return out

    @classmethod
    def from_store(cls, model, folder: str, model_name: Optional[str] = None, dtype: torch.dtype = torch.int16, **kw):
        """server.py:117-139: every shard of the store, BOS position dropped, resident on the model's device."""
        dev = next(model.parameters()).device
        name = model.name if model_name is None else model_name
        codes = store.load_code_shards(folder, name, skip_bos=True, dtype=dtype, device=dev)
        return cls(model, codes, **kw)

    # ------------------------------------------------------------------------------------------------
    def _query(self, idx, activation, n_layers: int) -> torch.Tensor:
        if activation is not None and idx is not None:
            raise ValueError("Cannot specify both idx and activation")
        elif idx is not None:
            q = self.activations[int(idx)]
        elif activation is not None:
            q = torch.as_tensor(activation)
        else:
            raise ValueError("Must specify either idx or activation")
        if q.dim() != 2 or q.shape[1] < n_layers:
            raise ValueError(f"query must be (positions, >= {n_layers} layers), got {tuple(q.shape)}")
        if q.shape[0] > SQ_PAD:
            raise NotImplementedError(f"at most {SQ_PAD} query positions (got {q.shape[0]})")
        return q[:, :n_layers].to(device=self.sims.device, dtype=torch.int32).contiguous()

    def accumulate(self, query: torch.Tensor, layers: Sequence[int]) -> Iterator[Tuple[torch.Tensor, torch.Tensor]]:
        """After every layer range of ``layers`` (server.py:198-263): (``intensity_accumulation`` as a view
        (N, S, Sq) of the padded fp16 buffer, per-position maxima (Sq, N) fp16 = ``max_values.T`` of :267).
        The buffers are reused from one step to the next, as in the reference."""
        layers = [int(l) for l in layers]
        if not layers or any(b <= a for a, b in zip([0] + layers[:-1], layers)):
            raise ValueError("layers must be strictly ascending positive layer indices")
        L = layers[-1]
        nq, K = self.sims.shape[0], self.sims.shape[1]
        N, S, nq_codes = self.activations.shape
        if L > nq or L > nq_codes:
            raise ValueError(f"max(layers)={L} exceeds the {min(nq, nq_codes)} layers of the table / code store")
        dev = self.sims.device
        Sq = query.shape[0]
        lib = _lib.load()
        # The device guard and the stream are taken around every group of C calls, never across a `yield`: the
        # consumer may switch device or stream between steps, and its own indexing of the yielded buffers runs on
        # whatever stream is current then.
        tbytes = lib.rqae_search_table_bytes(L, K)
        table = torch.empty(tbytes // 2, dtype=torch.float16, device=dev)
        with torch.cuda.device(dev):
            st = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(lib.rqae_search_build_table_f16(self.sims.data_ptr(), K, query.data_ptr(), query.stride(0), Sq, L,
                                                      table.data_ptr(), tbytes, st), "rqae_search_build_table_f16")
        last = torch.cuda.current_stream(dev)
        acc = torch.empty(N * S, SQ_PAD, dtype=torch.float16, device=dev)
        n_pad = (N + 7) // 8 * 8
        maxv = torch.empty(Sq, n_pad, dtype=torch.float16, device=dev)
        a = 0
        for b in layers:
            with torch.cuda.device(dev):
                cur = torch.cuda.current_stream(dev)
                if cur != last:          # the consumer changed streams: order this step after the previous one
                    cur.wait_stream(last)
                    for t in (table, acc, maxv, query):
                        t.record_stream(cur)
                    last = cur
                st = cur.cuda_stream
                _lib.check(lib.rqae_search_accumulate_f16(table.data_ptr(), K, self.activations.data_ptr(),
                                                         _lib.code_dtype(self.activations.dtype), nq_codes, N * S, a, b,
                                                         1 if a == 0 else 0, acc.data_ptr(), st), "rqae_search_accumulate_f16")
                _lib.check(lib.rqae_search_position_max_f16(acc.data_ptr(), N, S, Sq, maxv.data_ptr(), n_pad, st),
                           "rqae_search_position_max_f16")
            yield acc.view(N, S, SQ_PAD)[:, :, :Sq], maxv[:, :N]
            a = b

    def find_examples(self, idx: int = None, activation: torch.Tensor = None, top_examples: int = 30,
                      middle_examples: int = 10, bottom_examples: int = 10,
                      layers: List[int] = SERVER_LAYERS):
        """server.py:159-325."""
        layers = list(layers)
        query = self._query(idx, activation, max(layers))
        N = self.activations.shape[0]
        Sq = query.shape[0]
        k = window_k(top_examples, middle_examples, bottom_examples, N)
        from .feature import select_top_middle_bottom
        if self.precision == "tc":
            # every cut at once: one GEMM launch for the maxima, one selection launch over (cut, position) rows, one launch
            # for the exact rows of everything selected, two device->host copies; the generator then yields cut by cut
            maxv_all = self.maxima_tc(query, layers, padded=True)                      # (C, 128, N), rows >= Sq zero
            table = self._build_qrows(query, max(layers))
            sel, _ = select_top_middle_bottom(maxv_all, k, n=N)                        # (C, 128, 3, k) int32
            sel = sel[:, :Sq].contiguous()
            C = len(layers)
            lists = window_lists(sel.reshape(C * Sq, 3, k), top_examples, middle_examples, bottom_examples)
            names = list(lists)
            cat = torch.cat([lists[nm] for nm in names], dim=1).reshape(C, Sq, -1)     # (C, Sq, n_sel)
            rows_d = self.rows_exact(table, cat, layers, first_range=0)                # (C, Sq, n_sel, S)
            # per window one contiguous device tensor, one copy through a pinned staging buffer the engine keeps (a pageable
            # .cpu() of the 21 MB of rows costs 10 ms; allocating pinned memory per query costs as much on a cold process),
            # and one host copy out of it: what a cut yields is a contiguous view of that copy, owned by the caller
            stage, o = {}, 0
            for nm in names:
                w = lists[nm].shape[1]
                r_d, i_d = rows_d[:, :, o:o + w].contiguous(), cat[:, :, o:o + w].contiguous()
                r_h, i_h = self._pinned("rows_" + nm, r_d.shape, torch.float16), self._pinned("sel_" + nm, i_d.shape, torch.int32)
                r_h.copy_(r_d, non_blocking=True)
                i_h.copy_(i_d, non_blocking=True)
                stage[nm] = (i_h, r_h)
                o += w
            torch.cuda.current_stream(self.sims.device).synchronize()
            host = {nm: (stage[nm][0].clone(), stage[nm][1].clone()) for nm in names}
            for ci, layer in enumerate(layers):
                out = {nm: {"indices": host[nm][0][ci], "intensities": host[nm][1][ci]} for nm in names}
                yield out, layer
            return
        qpos = torch.arange(Sq, device=self.sims.device).unsqueeze(-1)
        for layer, (acc, maxv) in zip(layers, self.accumulate(query, layers)):
            sel, _ = select_top_middle_bottom(maxv, k, n=N)                  # (Sq, 3, k) int32
            out = {}
            for name, lst in window_lists(sel, top_examples, middle_examples, bottom_examples).items():
                inten = acc[lst.long(), :, qpos]                              # (Sq, k', S): intensity_accumulation[lst[i], :, i]
                out[name] = {"indices": lst.cpu().int(), "intensities": inten.cpu().to(torch.float16)}
            yield out, layer


def window_k(top_examples: int, middle_examples: int, bottom_examples: int, n_sequences: int) -> int:
    """The single window size the radix select is asked for: it returns argsort[:k], argsort[n//2 - k//2 : n//2 + k//2]
    and argsort[-k:]; the three lists of server.py:271-287 are sub-slices of those (``window_lists``)."""
    top, mid, bot = int(top_examples), int(middle_examples), int(bottom_examples)
    k = max(top, mid, bot, 1)
    if k > SELECT_KMAX:
        raise NotImplementedError(f"at most {SELECT_KMAX} examples per window")
    k = min(k, int(n_sequences))
    if mid // 2 > k // 2:
        raise ValueError(f"middle_examples={mid} needs at least {2 * (mid // 2)} sequences, the store has {n_sequences}")
    return k


def window_lists(sel: torch.Tensor, top_examples: int, middle_examples: int, bottom_examples: int) -> dict:
    """sel (Sq, 3, k) from the select -> {"top": (Sq, top), "middle": (Sq, 2*(mid//2)), "bottom": (Sq, bottom)},
    i.e. sorted[:top], sorted[n//2 - mid//2 : n//2 + mid//2], sorted[-bottom:] of server.py:271-287."""
    k = sel.shape[-1]
    top, mh, bot = min(int(top_examples), k), int(middle_examples) // 2, min(int(bottom_examples), k)
    kh = k // 2
    return {"top": sel[:, 0, :top], "middle": sel[:, 1, kh - mh: kh + mh], "bottom": sel[:, 2, k - bot:]}
