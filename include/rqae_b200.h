/*
 * rqae_b200 -- C ABI of the B200 (sm_100a) implementation of the RQAE residual-quantization
 * hot path.  Plain C: device pointers, sizes and a CUDA stream handle; no torch types.
 *
 * The reference (harish-kamath/rqae) is pure Python and has no FFI of its own; its boundary for
 * this path is the Python surface of `rqae.model.RQAE` (rqae/model.py).  Each entry point below
 * names the reference method it replaces.  `rqae_b200/model.py` is the reference-side binding
 * (ctypes), and INTEGRATION.md shows the three-line change a maintainer of the reference makes.
 *
 * Conventions
 *   - every function returns 0 on success or an RQAE_E* code; rqae_strerror() names it.
 *     No exception or signal crosses the ABI.  Asynchronous CUDA errors surface at the caller's
 *     next synchronisation, as with any kernel launch.
 *   - all `const float*` / `void*` data arguments are DEVICE pointers unless the name ends in
 *     `_host`.  The library never allocates or frees caller-visible memory; it borrows the
 *     pointers for the duration of the launch.
 *   - `stream` is a cudaStream_t passed as void* (0 = the legacy default stream).  Kernels are
 *     enqueued on it and the call returns without synchronising, so the functions can be called
 *     from inside a framework forward hook (rqae/model.py:276-289 runs mid-forward).
 *   - code tensors: `code_dtype` 0 = int16, 1 = int32, 2 = int64 (the reference returns int64,
 *     rqae/model.py:226; scripts/1_create_activations.py:184-186 stores int32).
 */
#ifndef RQAE_B200_H
#define RQAE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RQAE_OK 0
#define RQAE_EINVAL 1      /* bad argument (null pointer, non-positive size, unknown dtype) */
#define RQAE_EUNSUPPORTED 2 /* shape outside the compiled instantiations (codebook_dim != 4, dim > 3584) */
#define RQAE_ECUDA 3       /* a CUDA runtime call failed; see rqae_last_cuda_error() */
#define RQAE_ENODEVICE 4   /* no sm_100 device / kernels not loadable on the current device */
#define RQAE_ESIZE 5       /* caller's buffer is smaller than required */

#define RQAE_CODE_I16 0
#define RQAE_CODE_I32 1
#define RQAE_CODE_I64 2

/* Library / build identification ("rqae_b200 <version> sm_100a"). */
const char* rqae_version(void);
const char* rqae_strerror(int code);
/* cudaGetErrorString of the last failing CUDA call made by this library on this thread. */
const char* rqae_last_cuda_error(void);

/* Bytes of the packed weight buffer for a model with `nq` quantizer layers, hidden size `dim`,
 * `codebook_dim` (must be 4) and `K` codebook rows.  Returns 0 for unsupported shapes. */
size_t rqae_packed_bytes(int nq, int dim, int codebook_dim, int K);

/* Pack the weights of all layers into the streaming layout the kernels read (DESIGN.md).
 * Replaces nothing in the reference: it is the load-time step that follows
 * RQAE.load_state_dict (rqae/model.py:89-96).  Inputs are the reference parameters stacked
 * over layers, in the reference's own layouts:
 *   w_in  [nq][cd][dim]   layers.{l}.0.weight      b_in  [nq][cd]   layers.{l}.0.bias
 *   w_out [nq][dim][cd]   layers.{l}.1.weight      b_out [nq][dim]  layers.{l}.1.bias
 *   codebook [nq][K][cd] (codebook_shared = 0) or [1][K][cd] (= 1: fsq / round_fsq, where
 *   every layer holds the same table, rqae/model.py:63-72).
 * In shared mode bit-identical duplicate rows are removed from the search table (the lowest
 * original index is kept, which is what torch.argmax returns on ties). */
int rqae_pack_weights(const float* w_in, const float* b_in, const float* w_out, const float* b_out,
                      const float* codebook, int codebook_shared, int nq, int dim, int codebook_dim,
                      int K, void* packed, size_t packed_bytes, void* stream);

/* RQAE.forward (rqae/model.py:199-230), eval / temperature-0 semantics, all `nq_run` =
 * min(max_layers, nq) layers fused into one persistent kernel.
 *   x       [n_tokens][dim] fp32
 *   codes   [n_tokens][code_stride] of code_dtype, written for layers 0..nq_run-1 (nullable)
 *   q_out   [n_tokens][dim] fp32 reconstruction (nullable: "encode", codes only)
 *   teacher nullable int32 [n_tokens][nq_run]: codes that drive the residual recurrence while
 *           `codes` still receives this implementation's own per-layer argmax (parity testing)
 *   z_out   nullable fp32 [n_tokens][nq_run][4]: the in-projection values (parity testing)
 * `codebook` is the same device pointer that was given to rqae_pack_weights. */
int rqae_forward_f32(const void* packed, const float* codebook, int codebook_shared, int nq, int nq_run,
                     int dim, int codebook_dim, int K, const float* x, int64_t n_tokens, void* codes,
                     int code_dtype, int64_t code_stride, float* q_out, const int32_t* teacher,
                     float* z_out, void* stream);

/* Kernel variant of rqae_forward_f32 (process-wide): 0 (default) = one CTA per unit of tokens; 1 = where built (hidden
 * sizes 2305..3584), a cluster of two CTAs per unit, each owning half of the hidden dimension and exchanging its
 * in-projection partials through distributed shared memory.  The variants sum the in-projection in different orders
 * (both documented, both reproduced bit for bit by the C oracle), so codes can differ at near-ties; the variant is
 * therefore never switched implicitly.  Returns the previous setting (a negative argument only queries), or -1 for an
 * unknown variant.  Environment default: RQAE_CLUSTER=1. */
int rqae_forward_variant(int variant);

/* The body of RQAE.hook's hook_fn (rqae/model.py:276-289) for the Gemma-2 adapter (rqae/llm.py:60-73) in ONE launch:
 *     hs = hidden.float(); x = hs * rsqrt(mean(hs^2) + rms_eps) * (1 + rms_weight)          (llm.py:65-66)
 *     q, codes = forward(x)                                                                  (model.py:281)
 *     q = q / (1 + rms_weight) / rsqrt(mean(hs^2) + 1e-6)                                    (llm.py:68-73)
 *     q[:, 0] = hs[:, 0] when skip_bos (token t with t % seq_len == 0 is left untouched)     (model.py:285-286)
 *     hidden <- q in hidden's own dtype when replace                                         (model.py:289)
 * The normalisation, the de-normalisation, the BOS rule and the cast are fused into the load and the epilogue of
 * the forward kernel; no fp32 copy of the hidden states, no normalised copy and no fp32 reconstruction exist.
 *   hidden        [n_tokens][dim] of hidden_dtype (0 fp32, 1 fp16, 2 bf16), read and (replace != 0) overwritten
 *   rms_weight    fp32 [dim], the RMSNorm weight w (NOT 1 + w)
 *   codes         nullable, as in rqae_forward_f32
 * Arithmetic is fp32 with the reference's operation order; the sum of squares is accumulated in a different order
 * than torch's reduction, so results agree with the unfused path to fp32 rounding (codes: near-tie protocol). */
int rqae_hook_rmsnorm(const void* packed, const float* codebook, int codebook_shared, int nq, int nq_run, int dim,
                      int codebook_dim, int K, void* hidden, int hidden_dtype, int64_t n_tokens, int seq_len,
                      const float* rms_weight, float rms_eps, int skip_bos, int replace, void* codes, int code_dtype,
                      int64_t code_stride, void* stream);

/* RQAE.decode / decode_from_codebook_values (rqae/model.py:232-252): sum over the selected layers,
 * in ascending order, of W_out[l] c_l + b_out[l], with the reference's fp32 arithmetic
 * (o = fma(c3,w3,fma(c2,w2,fma(c1,w1,c0*w0))) + b; q = o_first, then q += o).
 *   codes       [n_tokens][code_stride] of code_dtype, or NULL when `cv` is given
 *   cv          nullable fp32 [n_tokens][nq][4] codebook values (decode_from_codebook_values)
 *   codebook0   [K][4] layer-0 table (the reference indexes codebook[0] for every layer)
 *   layer_mask  nullable uint8 [nq], DEVICE: 1 = include layer (the `layers=` filter)
 *   nq_codes    number of layers present in `codes` / `cv` (layers >= nq_codes are skipped) */
int rqae_decode_f32(const void* packed, const float* codebook0, int nq, int nq_codes, int dim,
                    int codebook_dim, int K, const void* codes, int code_dtype, int64_t code_stride,
                    const float* cv, const uint8_t* layer_mask, int64_t n_tokens, float* q_out,
                    void* stream);

/* Host-buffer front end of rqae_forward_f32 (the end-to-end path bench.py times as `e2e`):
 * x_host / codes_host / q_host are HOST pointers (pinned for full speed).  The call stages
 * chunks of `chunk_tokens` tokens through internal device buffers on three internal streams
 * (H2D, compute, D2H; three buffer sets) and returns after the last D2H copy has completed.
 * Every CUDA call on the way is checked; after a failure the streams are drained and RQAE_ECUDA
 * is returned.  The staging buffers, streams, events and worker threads are cached per calling
 * thread between calls; rqae_forward_host_release() frees them.
 *
 * rqae_forward_host_config selects how int32 / int64 codes reach `codes_host` (process-wide;
 * -1 keeps a setting):
 *   code_transfer  0 auto (= narrow), 1 narrow: int16 over PCIe into a pinned staging buffer, widened
 *                  into the caller's tensor by `widen_threads` host threads (a quarter of the PCIe
 *                  bytes; with 8 ranks on one host the device -> host bytes bound the rate, DESIGN.md 7);
 *                  2 direct: the kernel emits the caller's dtype and the copy lands in the caller's
 *                  tensor (no host threads, no staging)
 *   widen_threads  0 auto = cores / (2 * LOCAL_WORLD_SIZE), clamped to [1, 8]
 * Environment defaults: RQAE_HOST_CODES = auto | narrow | direct, RQAE_HOST_THREADS = n. */
int rqae_forward_host_f32(const void* packed, const float* codebook, int codebook_shared, int nq,
                          int nq_run, int dim, int codebook_dim, int K, const float* x_host,
                          int64_t n_tokens, void* codes_host, int code_dtype, float* q_host,
                          int64_t chunk_tokens);
int rqae_forward_host_config(int code_transfer, int widen_threads);
/* The settings in effect: *code_transfer = 1 narrow | 2 direct, *widen_threads = the resolved thread count. */
int rqae_forward_host_mode(int* code_transfer, int* widen_threads);
/* The widening step of the narrow mode on its own: int16 -> int32 / int64 with streaming stores on `threads`
 * host threads (0 = auto).  Host pointers; no CUDA call.  (scripts/1_create_activations.py:184-186 stores
 * int32: a caller that keeps int16 on the wire widens with this.) */
int rqae_widen_codes_host(const int16_t* src_host, void* dst_host, int64_t n, int code_dtype, int threads);
int rqae_forward_host_release(void);

/* RQAEFeature.intensity (rqae/feature.py:102-129) for `n_features` features at once -- the inner
 * computation of the mining loop scripts/3_make_rqae_features.py:98-114.  For feature f (center codes
 * centers[f][l]), token t and every cut c (cuts_host: strictly ascending layer indices, the
 * reference's `layers` list):
 *     out[f][c][t] = fp16( fp16( sum_{l<=cut} w_l * sims[center_f[l]][code_t[l]] ) / fp16( sum_{l<=cut} w_l ) )
 * with sims = codebook_sims (rqae/model.py:133-143) and w = the fp16 layer weights (feature.py:97-99).
 * Computed as one tcgen05 GEMM over the rank-4 factors of sims (DESIGN.md); the sum is accumulated in
 * fp32 from fp16 factors, so values agree with the reference within the tolerance DESIGN.md states,
 * not bitwise.  The roundings after the sum are the reference's.
 *   cb_norm            [K][4] fp32 = F.normalize(codebook[0], dim=-1)            (K + 1 <= 640)
 *   codes              [n_tokens][code_stride] of code_dtype (codes outside [0,K) contribute 0)
 *   centers            int32 [n_features][center_stride]
 *   layer_weights_f16  fp16 [>= max cut + 1]
 *   out                fp16 [n_features][n_cuts][out_stride]; out_stride >= n_tokens rounded up to a
 *                      multiple of 256 (whole token tiles are written), 16-byte aligned rows
 *   workspace          device scratch of rqae_intensity_workspace_bytes(...) bytes, 1024-byte aligned
 * Four launches on `stream` (schedule, code transpose, feature operand, GEMM); no synchronisation. */
size_t rqae_intensity_workspace_bytes(const int32_t* cuts_host, int n_cuts, int n_features, int64_t n_tokens);
int rqae_intensity_f16(const float* cb_norm, int K, const void* codes, int code_dtype, int64_t code_stride,
                       int64_t n_tokens, const int32_t* centers, int64_t center_stride, int n_features,
                       const void* layer_weights_f16, const int32_t* cuts_host, int n_cuts, void* out,
                       int64_t out_stride, void* workspace, size_t workspace_bytes, void* stream);
/* The same for another set of features over the SAME code tensor, cuts and codebook as the previous rqae_intensity_f16 call on
 * this workspace (scripts/3_make_rqae_features.py:164-196 mines its features group by group over one code store): the
 * tile-major copy of the codes is still in the workspace and is not rebuilt; the workspace must be large enough for this
 * call's n_features (rqae_intensity_workspace_bytes). */
int rqae_intensity_again_f16(const float* cb_norm, int K, int64_t n_tokens, const int32_t* centers, int64_t center_stride,
                             int n_features, const void* layer_weights_f16, const int32_t* cuts_host, int n_cuts, void* out,
                             int64_t out_stride, void* workspace, size_t workspace_bytes, void* stream);

/* Bit-exact RQAEFeature.intensity (rqae/feature.py:102-129) for `n_features` features at once: the reference's own
 * arithmetic, rounding for rounding (the opt-in exact path; rqae_intensity_f16 is the faster tolerance path).  For
 * feature f, token t and every cut (cuts_host: strictly ascending layer indices, deepest <= 4095, any number):
 *     p_l  = fp16( w_l * sims[centers[f][l]][codes[t][l]] )                    one rounding
 *     run  = +0.0f; run += float(p_l), l = 0, 1, ...       wrun likewise of float(w_l), both fp32, ascending layers
 *     out[f][c][t] = fp16( float(fp16(run)) / float(fp16(wrun)) )              IEEE fp32 divide
 * Code indexing is the reference's sims[center, codes]: a token or center code in [-K, 0) reads row code + K; a code
 * outside [-K, K), where the reference raises, contributes a +0 product.  (rqae_intensity_f16 treats every code
 * outside [0, K) as 0.)
 *   sims_f16           fp16 [K][K], the reference's codebook_sims (rqae/model.py:140-142), K < 640
 *   codes              [n_tokens][code_stride] of code_dtype, code_stride > deepest cut
 *   centers            int32 [n_features][center_stride], center_stride > deepest cut
 *   layer_weights_f16  fp16 [>= deepest cut + 1]; the weight prefixes are summed on the device
 *   out                fp16 [n_features][n_cuts][out_stride], out_stride >= n_tokens rounded up to 8 and a multiple
 *                      of 8, 16-byte aligned: the layout rqae_select_top_middle_bottom_f16 reads.  Only tokens
 *                      < n_tokens are written.
 * No workspace.  One launch on `stream` (none when n_tokens or n_features is 0); no synchronisation. */
int rqae_intensity_exact_f16(const void* sims_f16, int K, const void* codes, int code_dtype, int64_t code_stride,
                             int64_t n_tokens, const int32_t* centers, int64_t center_stride, int n_features,
                             const void* layer_weights_f16, const int32_t* cuts_host, int n_cuts, void* out,
                             int64_t out_stride, void* stream);

/* The selection step of the mining loop, scripts/3_make_rqae_features.py:116-128: for every row
 * (one feature at one cut) of `vals`, the positions of the top_k largest values, of the 2*(top_k/2)
 * values around the median rank and of the top_k smallest, i.e. argsort(descending)[:k],
 * [n/2 - k/2 : n/2 + k/2] and [-k:], by an exact radix select instead of a full sort.  Total order:
 * value descending, index ascending (the reference's argsort leaves ties unspecified).
 *   vals     fp16 [rows][row_stride], 16-byte aligned rows (row_stride % 8 == 0), readable up to n
 *            rounded up to 8 -- the layout rqae_intensity_f16 writes
 *   idx_out  int32 [rows][3][top_k] (top, middle, bottom), -1 in unused middle slots
 *   val_out  nullable fp16 [rows][3][top_k], the selected values
 * top_k <= 256, top_k <= n < 2^31.
 * Rows of 16 384 .. 262 144 values go through the sample-bracketed single-pass kernel (rq_mine3.cuh); a row whose
 * brackets miss, and every other row length, through the three-pass kernel (rq_mine.cuh) -- same result, same order.
 * The call takes a few bytes per row from a stream-ordered pool of the library (cudaMallocFromPoolAsync on `stream`) for the
 * fallback list.  Environment, read per call: RQAE_MINE_V2=1 runs the three-pass kernel for every row (A/B timing of
 * the two kernels; the only selection switch). */
int rqae_select_top_middle_bottom_f16(const void* vals, int64_t rows, int64_t row_stride, int64_t n, int top_k,
                                      int32_t* idx_out, void* val_out, void* stream);

/* Nearest-example search over a code store: the inner loops of IntensityEngine.find_examples
 * (demo/server/server.py:159-325), split at the points where the reference hands data between steps.
 * `sims_f16` is the engine's table (server.py:104-115): fp16 [nq][K][K] = subfeature_sims * layer_norms, indexed
 * [layer][query code][dataset code].  All roundings are the reference's (fp16 table values, fp32 sum inside a chunk
 * of <= 64 layers rounded to fp16, fp16 adds between chunks and between layer ranges); the only freedom is the order
 * of the fp32 additions inside a chunk (ascending layer order here).
 *
 * rqae_search_build_table_f16 -- server.py:176-196: the query's rows of the table for layers [0, n_layers),
 *   table[l][c][q] = sims[l][query[q][l]][c], fp16 [n_layers][K][128], q >= n_query zero-filled (one 256-byte row
 *   per (layer, dataset code)).   query: int32 [n_query][query_stride], n_query <= 128; a query code outside [0,K)
 *   gives a zero row.  table_bytes >= rqae_search_table_bytes(n_layers, K); 16-byte aligned.
 * rqae_search_accumulate_f16 -- server.py:41-68 (get_intensities), :204-263: for every dataset token t,
 *   acc[t][q] (+)= sum over layers [layer_begin, layer_end) of table[l][codes[t][l]][q]   (one layer range of the
 *   reference's `layers` list per call; `first` != 0 stores instead of adding: the reference's first range).
 *   codes [n_tokens][code_stride] of code_dtype, tokens sequence-major (token = sequence * seq_len + position);
 *   acc fp16 [n_tokens][128] = the reference's intensity_accumulation (N, S, Sq) with Sq padded to 128.
 *   A dataset code outside [0,K) contributes 0 (the reference would raise an indexing error).
 * rqae_search_position_max_f16 -- server.py:265-267: out[q][n] = max over the seq_len positions of sequence n of
 *   acc[n*seq_len + s][q] (a NaN wins, as in torch.max), fp16 [n_query][out_stride], out_stride % 8 == 0,
 *   out_stride >= n_seq, columns >= n_seq zero-filled: the row layout rqae_select_top_middle_bottom_f16 reads, which
 *   then replaces the argsort + slices of server.py:268-287. */
size_t rqae_search_table_bytes(int n_layers, int K);
int rqae_search_build_table_f16(const void* sims_f16, int K, const int32_t* query, int64_t query_stride, int n_query,
                                int n_layers, void* table, size_t table_bytes, void* stream);
int rqae_search_accumulate_f16(const void* table, int K, const void* codes, int code_dtype, int64_t code_stride,
                               int64_t n_tokens, int layer_begin, int layer_end, int first, void* acc, void* stream);
int rqae_search_position_max_f16(const void* acc, int64_t n_seq, int seq_len, int n_query, void* out,
                                 int64_t out_stride, void* stream);

/* Opt-in tensor-core variant of RQAE.decode (rqae/model.py:232-252): the same sum as rqae_decode_f32,
 * evaluated as one tcgen05 GEMM  q[t][d] = sum_{l,j} V[t][4l+j] * U[d][4l+j] + sum_l b_out[l][d]  with
 * V = codebook[0][codes] and U = W_out, fp16 operands and fp32 accumulation.  NOT bit-exact (the default
 * rqae_decode_f32 is): `passes` = 1 rounds both operands to fp16 (relative error of q about 3e-4),
 * `passes` = 3 adds the fp16 remainders of both operands (V_hi U_hi + V_hi U_lo + V_lo U_hi: about 2e-5,
 * which is the tensor core's own fp32 accumulation over 12 288 terms, no longer the operand rounding).
 *   w_out [nq][dim][4] and b_out [nq][dim]: the reference parameters stacked over layers (layers.{l}.1.*)
 *   codebook0 [K][4], K + 1 <= 640; codes / code_dtype / code_stride / layer_mask / nq_codes as in rqae_decode_f32
 *   workspace: device scratch of rqae_decode_tc_workspace_bytes(...) bytes, 1024-byte aligned
 * nq_codes * passes <= 3200 layers-passes (200 K-blocks of 16 layers). */
size_t rqae_decode_tc_workspace_bytes(int nq_codes, int dim, int64_t n_tokens, int passes);
int rqae_decode_tc_f32(const float* w_out, const float* b_out, const float* codebook0, int nq, int nq_codes, int dim,
                       int codebook_dim, int K, const void* codes, int code_dtype, int64_t code_stride,
                       const uint8_t* layer_mask, int64_t n_tokens, float* q_out, int passes, void* workspace,
                       size_t workspace_bytes, void* stream);

/* Measurement helpers used by bench.py for the roofline denominators (no model semantics):
 * sustained rate of the FP32 pipe, in FLOP per call; time it with CUDA events on `stream`.
 *   packed_f32x2 = 1  dense FFMA2 (the peak the roofline fraction is quoted against)
 *                = 0  scalar FFMA
 *                = 2  the operand pattern of the forward kernel's in-projection sweep
 *                     (scalar weight x token pair + pair accumulator), registers only
 *                = 3  the pattern of its out-projection sweep (fma chain over k, residual update)
 * Modes 2/3 read `sink[64..191]` as data (fill >= 192 floats) and show what the register file lets
 * the FMA pipe deliver for the kernel's instruction mix (DESIGN.md, 4.1). */
int rqae_fp32_peak_probe(int packed_f32x2, int iters, double* flops_per_launch, float* sink, void* stream);

/* Tensor-core form of the search maxima (opt-in, NOT bit-exact; replaces the accumulate + per-position max of
 * demo/server/server.py:204-267 for the RANKING only).  The engine's table is rank 5 per layer, so the accumulation is a
 * GEMM over (layer, factor) with fp16 factor tables: vtab[l][c] = the dataset-side factor of codeword c at layer l,
 * utab[l][c] = the same times the layer norm (query side), both [table_layers][640] rows of 8 fp16 (5 used; row K and
 * the layers beyond the model's zero; table_layers a multiple of 8).
 *   rqae_search_tc_pack_store   code store (n_seq, seq_len <= 128, code_stride) -> the 8-layer block-major copy the GEMM
 *                               streams (once per store, not per query)
 *   rqae_search_tc_maxima_f16   for every range end of `layers_host` (the `layers` list of find_examples):
 *                               max_out[(c * 128 + q) * max_stride + n] = fp16(max_s sum_{l < layers[c]} table entry),
 *                               rows = what rqae_select_top_middle_bottom_f16 ranks (row stride max_stride, n = n_seq)
 *   rqae_search_rows_f16        rows_out[c][q][j][s] = intensity_accumulation[sel[c][q][j], s, q] after the ranges
 *                               0 .. first_range + c of layers_host, c < n_cuts (one launch serves the selections of
 *                               several consecutive cuts), with the reference's exact arithmetic (the rounding points of
 *                               rqae_search_accumulate_f16), from `table` = the query's rows of the engine table as
 *                               they lie, Qr[l][q][c] = sims[l][query[q][l]][c] (rqae_search_build_qrows_f16;
 *                               server.py:183-196's query_sims): server.py:290-305 for the selected sequences only. */
size_t rqae_search_tc_store_bytes(int64_t n_seq, int nq_codes);
size_t rqae_search_qrows_bytes(int n_layers, int n_query, int K);
int rqae_search_build_qrows_f16(const void* sims_f16, int K, const int32_t* query, int64_t query_stride, int n_query,
                                int n_layers, void* qrows, size_t qrows_bytes, void* stream);
int rqae_search_tc_pack_store(const void* codes, int code_dtype, int64_t code_stride, int64_t n_seq, int seq_len,
                              int nq_codes, int K, void* store_tc, size_t store_bytes, void* stream);
size_t rqae_search_tc_workspace_bytes(const int32_t* layers_host, int n_layers_list);
int rqae_search_tc_maxima_f16(const void* store_tc, int64_t n_seq, int seq_len, int nq_codes, const void* vtab_f16,
                              const void* utab_f16, int table_layers, int K, const int32_t* query, int64_t query_stride,
                              int n_query, const int32_t* layers_host, int n_layers_list, void* max_out, int64_t max_stride,
                              void* workspace, size_t workspace_bytes, void* stream);
int rqae_search_rows_f16(const void* table, int K, const void* codes, int code_dtype, int64_t code_stride, int64_t n_seq,
                         int seq_len, const int32_t* sel, int n_query, int n_sel, const int32_t* layers_host,
                         int first_range, int n_cuts, void* rows_out, void* stream);

/* Number of kernels this library has launched on this thread since the last reset
 * (bench.py reports it as gpu_launches). */
int64_t rqae_launch_count(int reset);

#ifdef __cplusplus
}
#endif
#endif /* RQAE_B200_H */
