// Nearest-example search over a code store (sm_100a) -- SURVEY 8f-3.
//
// Replaces the inner loops of IntensityEngine.find_examples (reference harish-kamath/rqae,
// demo/server/server.py:159-325).  For a query of Sq <= 128 positions and a dataset of N sequences of S
// positions, the reference keeps  intensity_accumulation[n][s][q] (fp16)  and, for every layer range
// [a, b) of its `layers` list, adds
//     sum_{l in [a,b)} sims[l][ q_code[q][l] ][ d_code[n][s][l] ]                 (server.py:41-68, 204-263)
// where sims = subfeature_sims * layer_norms is an fp16 table (server.py:104-115).  The reference
// materialises the gathered values as a (1024, 127, 127, <=64) fp16 tensor per shard and chunk (2.1 GB) and
// reduces it with `sum(dim=-1)`; here the gather, the sum and the accumulation are one pass:
//
//   search_table_kernel       Qt[l][c][q] = sims[l][q_code[q][l]][c], q padded to 128 with zeros: the
//                             query's rows of the table, transposed so that everything one dataset token
//                             needs at one layer is ONE contiguous 256-byte row (server.py:183-196 builds
//                             the same rows untransposed)
//   search_accumulate_kernel  a warp owns 8 dataset tokens; lane j owns query positions 4j..4j+3; per
//                             (token, layer) one coalesced 256-byte row load from L1/L2 and four fp32 adds
//                             per lane.  Roundings are the reference's: fp32 running sum inside a chunk of
//                             <= 64 layers (ascending layer order), one rounding to fp16 per chunk, chunks
//                             of a range added in fp16 (server.py:216-234), ranges added in fp16 (:256-259)
//   search_posmax_kernel      max over the S positions of every dataset sequence (server.py:265-267),
//                             written query-position-major so that the selection (rq_mine.cuh) can rank the
//                             sequences of every query position without the reference's full argsort
//
// Bound: the table rows.  A token-layer reads 256 B of table against 2-4 B of code store, and a layer's slab
// (K x 256 B = 160 KB at K = 625) is as large as an SM's L1 (hit rate 9 %), so the rows come from L2: the kernel
// runs at the rate L2 delivers 256-byte rows to the SMs (6.2-7.6 TB/s measured), not at the HBM rate of the code
// store (DESIGN.md 4.6 has the arithmetic, the measurements and the plan).
#pragma once
#include <cuda_fp16.h>

#include "rq_common.cuh"
#include "rq_intensity.cuh"

namespace rq {

constexpr int SR_Q = 128;            // padded query positions (row = 128 fp16 = 256 B)
constexpr int SR_THREADS = 256;      // accumulate kernel: 8 warps
constexpr int SR_TOK_PER_WARP = 8;
constexpr int SR_TILE = (SR_THREADS / 32) * SR_TOK_PER_WARP;   // 64 tokens per CTA pass
constexpr int SR_CHUNK = 64;         // server.py:219-222: a range longer than 64 layers is summed in chunks of 64

// ---------------------------------------------------------------------------------------------------------
// Qt[l][c][q] = sims[l][qcode[q][l]][c]
// ---------------------------------------------------------------------------------------------------------
struct SearchTableParams {
  const __half* sims;       // [>= n_layers][K][K]
  const int* query;         // [n_query][query_stride] int32 codes
  long long query_stride;
  int n_query, n_layers, K;
  __half* table;            // [n_layers][K][SR_Q]
};

__global__ void __launch_bounds__(256) search_table_kernel(const SearchTableParams p) {
  __shared__ __half tile[SR_Q][34];
  const int l = blockIdx.y, c0 = blockIdx.x * 32, tid = threadIdx.x;
  const int K = p.K;
  {
    const int cc = tid & 31, qq = tid >> 5;
    for (int q = qq; q < SR_Q; q += 8) {
      __half v = __float2half(0.f);
      if (q < p.n_query && c0 + cc < K) {
        const int qc = p.query[(long long)q * p.query_stride + l];
        if (qc >= 0 && qc < K) v = p.sims[((size_t)l * K + qc) * K + c0 + cc];
      }
      tile[q][cc] = v;
    }
  }
  __syncthreads();
  {
    const int q = tid & (SR_Q - 1), ch = tid >> 7;
    for (int cc = ch; cc < 32; cc += 2)
      if (c0 + cc < K) p.table[((size_t)l * K + c0 + cc) * SR_Q + q] = tile[q][cc];
  }
}

// ---------------------------------------------------------------------------------------------------------
// acc[t][q] (+)= range sum
// ---------------------------------------------------------------------------------------------------------
struct SearchAccParams {
  const __half* table;      // [.. layer_end][K][SR_Q]
  const void* codes;        // [n_tokens][code_stride] of CodeT
  long long code_stride, n_tokens;
  int K, layer_begin, layer_end, first;
  __half* acc;              // [n_tokens][SR_Q]
};

__device__ __forceinline__ uint32_t sr_pack(float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ float2 sr_unpack(uint32_t w) { return __half22float2(*reinterpret_cast<const __half2*>(&w)); }

template <typename CodeT>
__global__ void __launch_bounds__(SR_THREADS, 2) search_accumulate_kernel(const SearchAccParams p) {
  // DEPTH = layers of row loads kept in flight per token: the loads of layer i + DEPTH are issued as soon as layer i
  // has been consumed (DEPTH x 8 independent 256-byte rows outstanding per warp).  Measured on the whole store,
  // DEPTH 1 / 2 / 3 = 197 / 196 / 275 ms (profiles/r1s_search_ab.jsonl): the kernel is bound by what L2 delivers, not
  // by the latency a warp sees, so 2 rides out the DRAM misses of the longest range and 3 only adds queueing.
  constexpr int DEPTH = 2;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const CodeT* __restrict__ codes = (const CodeT*)p.codes;
  const long long n_tiles = (p.n_tokens + SR_TILE - 1) / SR_TILE;
  const int K = p.K;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long tok0 = tile * SR_TILE + warp * SR_TOK_PER_WARP;
    if (tok0 >= p.n_tokens) continue;
    uint32_t rng[SR_TOK_PER_WARP][2];       // the range's value so far: four fp16 per token, packed
    for (int c0 = p.layer_begin; c0 < p.layer_end; c0 += SR_CHUNK) {
      const int c1 = (c0 + SR_CHUNK < p.layer_end) ? c0 + SR_CHUNK : p.layer_end;
      float cs[SR_TOK_PER_WARP][4];
#pragma unroll
      for (int j = 0; j < SR_TOK_PER_WARP; ++j) cs[j][0] = cs[j][1] = cs[j][2] = cs[j][3] = 0.f;
      for (int l0 = c0; l0 < c1; l0 += 32) {
        const int nl = (c1 - l0 < 32) ? c1 - l0 : 32;
        int mine[SR_TOK_PER_WARP];          // lane i holds the codes of layer l0 + i
#pragma unroll
        for (int j = 0; j < SR_TOK_PER_WARP; ++j) {
          mine[j] = -1;
          if (lane < nl && tok0 + j < p.n_tokens) {
            const long long v = (long long)codes[(tok0 + j) * p.code_stride + l0 + lane];
            mine[j] = (v >= 0 && v < K) ? (int)v : -1;
          }
        }
        const __half* slab0 = p.table + (size_t)l0 * K * SR_Q + 4 * lane;
        uint2 w[DEPTH][SR_TOK_PER_WARP];
        // issue the eight row loads of layer l0 + i into buffer b
#define SR_ISSUE(b, i)                                                                              \
  {                                                                                                 \
    const __half* slab = slab0 + (size_t)(i) * K * SR_Q;                                            \
    _Pragma("unroll") for (int j = 0; j < SR_TOK_PER_WARP; ++j) {                                   \
      const int c = __shfl_sync(0xffffffffu, mine[j], (i)); /* warp-uniform */                      \
      w[b][j] = make_uint2(0u, 0u); /* a code outside [0, K) or a token past the end adds +0 */     \
      if (c >= 0) w[b][j] = __ldg(reinterpret_cast<const uint2*>(slab + (size_t)c * SR_Q));         \
    }                                                                                               \
  }
#pragma unroll
        for (int d = 0; d < DEPTH; ++d)
          if (d < nl) SR_ISSUE(d, d)
        for (int i = 0; i < nl; i += DEPTH) {
#pragma unroll
          for (int d = 0; d < DEPTH; ++d) {
            if (i + d < nl) {
#pragma unroll
              for (int j = 0; j < SR_TOK_PER_WARP; ++j) {
                const float2 lo = sr_unpack(w[d][j].x), hi = sr_unpack(w[d][j].y);
                cs[j][0] += lo.x; cs[j][1] += lo.y; cs[j][2] += hi.x; cs[j][3] += hi.y;   // ascending layer order
              }
              if (i + d + DEPTH < nl) SR_ISSUE(d, i + d + DEPTH)
            }
          }
        }
#undef SR_ISSUE
      }
#pragma unroll
      for (int j = 0; j < SR_TOK_PER_WARP; ++j)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const uint32_t h = sr_pack(cs[j][2 * e], cs[j][2 * e + 1]);              // sum(dim=-1) of an fp16 tensor
          if (c0 == p.layer_begin) {
            rng[j][e] = h;
          } else {                                                                 // intensities += chunk (fp16)
            const float2 a = sr_unpack(rng[j][e]), b = sr_unpack(h);
            rng[j][e] = sr_pack(a.x + b.x, a.y + b.y);
          }
        }
    }
#pragma unroll
    for (int j = 0; j < SR_TOK_PER_WARP; ++j) {
      if (tok0 + j >= p.n_tokens) break;
      uint2* dst = reinterpret_cast<uint2*>(p.acc + (size_t)(tok0 + j) * SR_Q + 4 * lane);
      uint2 r = make_uint2(rng[j][0], rng[j][1]);
      if (!p.first) {                                                              // intensity_accumulation += range (fp16)
        const uint2 o = *dst;
        const float2 a0 = sr_unpack(o.x), b0 = sr_unpack(r.x), a1 = sr_unpack(o.y), b1 = sr_unpack(r.y);
        r.x = sr_pack(a0.x + b0.x, a0.y + b0.y);
        r.y = sr_pack(a1.x + b1.x, a1.y + b1.y);
      }
      *dst = r;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// out[q][n] = max_s acc[n * S + s][q]
// ---------------------------------------------------------------------------------------------------------
struct SearchMaxParams {
  const __half* acc;        // [n_seq * seq_len][SR_Q]
  long long n_seq, out_stride;
  int seq_len, n_query;
  __half* out;              // [n_query][out_stride]; columns n_seq..out_stride-1 are zero-filled
};

__device__ __forceinline__ float sr_max_nan(float m, float v) { return (v > m || v != v) ? v : m; }   // torch.max: a NaN wins and stays

// 32 sequences per CTA; a warp takes four of them in turn and reads whole 256-byte rows (lane = 4 query positions).
__global__ void __launch_bounds__(256) search_posmax_kernel(const SearchMaxParams p) {
  __shared__ __half tile[32][SR_Q + 2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long n0 = (long long)blockIdx.x * 32;
  for (int k = 0; k < 4; ++k) {
    const int nl = warp * 4 + k;
    const long long n = n0 + nl;
    float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f;
    if (n < p.n_seq) {
      const uint2* src = reinterpret_cast<const uint2*>(p.acc + (size_t)n * p.seq_len * SR_Q) + lane;
      {
        const uint2 w = src[0];
        const float2 lo = sr_unpack(w.x), hi = sr_unpack(w.y);
        m0 = lo.x; m1 = lo.y; m2 = hi.x; m3 = hi.y;
      }
#pragma unroll 4
      for (int s = 1; s < p.seq_len; ++s) {
        const uint2 w = src[(size_t)s * (SR_Q / 4)];
        const float2 lo = sr_unpack(w.x), hi = sr_unpack(w.y);
        m0 = sr_max_nan(m0, lo.x); m1 = sr_max_nan(m1, lo.y); m2 = sr_max_nan(m2, hi.x); m3 = sr_max_nan(m3, hi.y);
      }
    }
    tile[nl][4 * lane + 0] = __float2half_rn(m0);
    tile[nl][4 * lane + 1] = __float2half_rn(m1);
    tile[nl][4 * lane + 2] = __float2half_rn(m2);
    tile[nl][4 * lane + 3] = __float2half_rn(m3);
  }
  __syncthreads();
  {
    const int nl = tid & 31, qq = tid >> 5;
    const long long n = n0 + nl;
    if (n < p.out_stride)
      for (int q = qq; q < p.n_query; q += 8) p.out[(size_t)q * p.out_stride + n] = tile[nl][q];
  }
}

// ---------------------------------------------------------------------------------------------------------
// Tensor-core form of the per-position maxima (opt-in, not bit-exact; DESIGN.md 4.6)
// ---------------------------------------------------------------------------------------------------------
// The engine's table is rank 5 per layer: subfeature_sims[l][a][b] is the cosine of the affine images of two codewords
// (rqae/model.py:145-167), i.e. f_l(a) . f_l(b) with unit 5-vectors f_l(c), and server.py:104-115 scales it by the layer
// norm.  Hence  acc[t][q] = sum_l  F_l[code_t[l]] . (norm_l F_l[qcode_q[l]])  is a dense contraction over k = (l, j):
// rq_intensity_kernel<2> runs it on the tensor cores with the dataset operand gathered per (token, layer) as ONE
// 16-byte row (5 values padded to 8) from a 10 MB table instead of the exact kernel's 256-byte row of table entries,
// keeps the running fp32 prefix in TMEM, and at every cut writes only max over the positions of each sequence.
// What differs from the reference: the products are not rounded to fp16 table entries and the prefix is not rounded
// per chunk / range, so a maximum can sit a few fp16 steps from the reference's (tests state the bound); the rows
// reported for the selected sequences are recomputed exactly by search_rows_kernel below.

// code store (n_seq, seq_len, stride) -> [n_units][L8][256] rows of 8 int16 codes: unit u holds sequences 2u and 2u+1
// in rows 0..127 / 128..255 (row = position); out-of-range codes, missing positions / sequences / layers -> K (zero row)
template <typename CT>
__global__ void __launch_bounds__(256) srch_pack_store_kernel(const CT* __restrict__ codes, long long stride, long long n_seq,
                                                              int seq_len, int n_layers, int K, int L8, uint4* __restrict__ out) {
  const long long u = blockIdx.x;
  const int r = threadIdx.x;
  const long long seq = 2 * u + (r >> 7);
  const int pos = r & 127;
  const bool live = seq < n_seq && pos < seq_len;
  const CT* src = codes + (live ? (seq * seq_len + pos) * stride : 0);
  for (int j = blockIdx.y; j < L8; j += gridDim.y) {
    uint32_t w[4];
#pragma unroll
    for (int h = 0; h < 4; h++) {
      uint32_t pr[2];
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const int l = 8 * j + 2 * h + e;
        uint32_t v = (uint32_t)K;
        if (live && l < n_layers) {
          const long long c = (long long)src[l];
          if (c >= 0 && c < K) v = (uint32_t)c;
        }
        pr[e] = v;
      }
      w[h] = pr[0] | (pr[1] << 16);
    }
    out[((size_t)u * L8 + j) * 256 + r] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

struct SrchPrepParams {
  int ends[IT_MAX_CUTS];   // the `layers` list: range c is [ends[c-1], ends[c])
  int n_cuts;
  IntKBlock* sched;        // entry: l0 = 8-layer block index, n = lo | hi << 8 (layers [lo, hi) of the block belong to the
};                         // segment: the query operand is zero outside), cut >= 0 on the last entry of a segment

__global__ void srch_prep_kernel(const SrchPrepParams p) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  int kb = 0, a = 0;
  for (int c = 0; c < p.n_cuts; c++) {
    const int b = p.ends[c];
    for (int j = a / 8; j <= (b - 1) / 8; j++) {
      IntKBlock e;
      const int lo = max(a, 8 * j) - 8 * j, hi = min(b, 8 * j + 8) - 8 * j;
      e.l0 = j; e.n = lo | (hi << 8); e.cut = (j == (b - 1) / 8) ? c : -1; e.tab = 0;
      p.sched[kb++] = e;
    }
    a = b;
  }
}

// query operand tiles: [NKB] tiles of 128 query positions x 64 k fp16 (8 layers x 8), swizzled like the feature tiles;
// row q, layer i of entry kb = utab[8 j + i][qcode[q][8 j + i]] inside the entry's layer window, else zero
__global__ void srch_pack_u_kernel(const int* __restrict__ query, long long query_stride, int n_query, int n_layers, int K,
                                   const uint4* __restrict__ utab, const IntKBlock* __restrict__ sched, int NKB,
                                   unsigned char* __restrict__ u_tiles) {
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= NKB * IT_FT * 8) return;
  const int i = gid & 7, q = (gid >> 3) & (IT_FT - 1), kb = gid >> 10;
  const IntKBlock e = sched[kb];
  const int lo = e.n & 0xFF, hi = e.n >> 8, l = 8 * e.l0 + i;
  uint4 v = make_uint4(0u, 0u, 0u, 0u);
  if (q < n_query && i >= lo && i < hi && l < n_layers) {
    const int c = query[(long long)q * query_stride + l];
    if (c >= 0 && c < K) v = __ldg(utab + (size_t)l * IT_LUT_ROWS + c);
  }
  *reinterpret_cast<uint4*>(u_tiles + (size_t)kb * IT_U_TILE + q * 128 + ((i ^ (q & 7)) << 4)) = v;
}

// ---------------------------------------------------------------------------------------------------------
// rows[q][j][s] = intensity_accumulation[sel[q][j], s, q] after the ranges ends[0..n_ranges), recomputed with the
// reference's arithmetic (the roundings of search_accumulate_kernel) for the selected sequences only
// (server.py:290-305).  One warp per (query position, selected sequence); lanes take the positions.
// ---------------------------------------------------------------------------------------------------------
// Qr[l][q][c] = sims[l][qcode[q][l]][c]: the query's rows of the table as they lie (server.py:183-196's `query_sims`).
// The rows kernel below gathers from THIS layout: for one (layer, query position) all K entries are 1 250 contiguous
// bytes, so the warps that work on the same query position (a block holds eight selected sequences of one position) find
// each other's sectors in L1; from the code-major table of the accumulate kernel every gather was a sector of its own.
__global__ void __launch_bounds__(256) search_qrows_kernel(const __half* __restrict__ sims, const int* __restrict__ query,
                                                           long long query_stride, int n_query, int n_layers, int K,
                                                           __half* __restrict__ out) {
  const int l = blockIdx.y, q = blockIdx.x;
  if (l >= n_layers || q >= n_query) return;
  const int qc = query[(long long)q * query_stride + l];
  __half* dst = out + ((size_t)l * n_query + q) * K;
  const __half* src = sims + ((size_t)l * K + (qc >= 0 && qc < K ? qc : 0)) * K;
  const bool ok = qc >= 0 && qc < K;
  for (int c = threadIdx.x; c < K; c += blockDim.x) dst[c] = ok ? src[c] : __float2half(0.f);
}

struct SearchRowsParams {
  const __half* table;      // Qr [layers][n_query][K]
  const void* codes;        // [n_seq][seq_len][code_stride]
  long long code_stride, n_seq;
  int seq_len, K, n_query, n_sel, n_cuts;   // n_cuts selections of [n_query][n_sel] sequences; selection c uses ranges 0 .. first_range + c
  int first_range;
  int ends[IT_MAX_CUTS];
  const int* sel;           // [n_cuts][n_query][n_sel] sequence indices (< 0: skipped, the row is zero-filled)
  __half* out;              // [n_cuts][n_query][n_sel][seq_len]
};

// One block per (cut, query position): its selected sequences all read the same table rows Qr[l][q][:], so the block
// stages the rows of 16 layers (20 KB) in shared memory and every thread advances its items -- (selected sequence,
// position) pairs, up to SRW_ITEMS per thread -- through them; fp32 chunk sums and the fp16 range / accumulation values
// of the items stay in registers.  (A warp per pair gathering two-byte entries straight from L1 was bound by the L1
// data pipe: 7.7 ms for the 82 550 pairs of a query; 13 ms from the code-major table.)
constexpr int SRW_THREADS = 256;
constexpr int SRW_ITEMS = 26;                        // items per thread and pass: 6 656 per block (50 selections x 127 positions = 6 350)
constexpr int SRW_PASS = SRW_THREADS * SRW_ITEMS;
constexpr int SRW_KMAX = 640;                        // table row length the staging buffer holds
constexpr int SRW_LB = 16;                           // layers per stage: an item's codes of a stage are one whole 32-byte sector (static shared memory: 47 KB)

template <typename CodeT>
__global__ void __launch_bounds__(SRW_THREADS) search_rows_kernel(const SearchRowsParams p) {
  __shared__ __align__(16) __half tab[SRW_LB][SRW_KMAX];
  __shared__ uint32_t tok[SRW_PASS];                 // token index (sequence * seq_len + position) of every item, 0xFFFFFFFF: skipped
  const int tid = threadIdx.x;
  const int cut = p.n_cuts - 1 - blockIdx.x / p.n_query, q = blockIdx.x % p.n_query;   // deepest cuts first: their blocks run longest
  const int n_ranges = p.first_range + cut + 1;
  const int K = p.K;
  const long long per = (long long)p.n_sel * p.seq_len;
  const int* sel = p.sel + ((size_t)cut * p.n_query + q) * p.n_sel;
  __half* out = p.out + ((size_t)cut * p.n_query + q) * (size_t)per;
  const CodeT* __restrict__ codes = (const CodeT*)p.codes;
  const __half* __restrict__ qr = p.table + (size_t)q * K;
  const size_t lstride = (size_t)p.n_query * K;
  // int16 code rows that start on 16-byte boundaries: the 8 codes of an aligned layer block are one vector load
  const bool vec16 = sizeof(CodeT) == 2 && (p.code_stride % SRW_LB) == 0 && ((uintptr_t)p.codes % 32) == 0;
  for (long long base = 0; base < per; base += SRW_PASS) {
    for (int i = tid; i < SRW_PASS; i += SRW_THREADS) {
      const long long it = base + i;
      uint32_t t = 0xFFFFFFFFu;
      if (it < per) {
        const int j = (int)(it / p.seq_len), s = (int)(it - (long long)j * p.seq_len);
        const long long n = sel[j];
        if (n >= 0 && n < p.n_seq) t = (uint32_t)(n * p.seq_len + s);
      }
      tok[i] = t;
    }
    __syncthreads();
    float cs[SRW_ITEMS];
    __half rng[SRW_ITEMS], acc[SRW_ITEMS];
#pragma unroll
    for (int k = 0; k < SRW_ITEMS; k++) { cs[k] = 0.f; rng[k] = __float2half(0.f); acc[k] = __float2half(0.f); }
    int a = 0;
    for (int r = 0; r < n_ranges; r++) {
      const int b = p.ends[r];
      for (int c0 = a; c0 < b; c0 += SR_CHUNK) {
        const int c1 = (c0 + SR_CHUNK < b) ? c0 + SR_CHUNK : b;
        for (int jb = c0 / SRW_LB; jb <= (c1 - 1) / SRW_LB; jb++) {            // aligned blocks of SRW_LB layers: the codes of an item are whole 32-byte sectors
          const int l0 = SRW_LB * jb;
          const int lo = (c0 > l0 ? c0 : l0) - l0, hi = (c1 < l0 + SRW_LB ? c1 : l0 + SRW_LB) - l0;
          __syncthreads();                                                    // the previous stage has been consumed
          for (int i = tid; i < (hi - lo) * K; i += SRW_THREADS) {
            const int li = i / K, c = i - li * K;
            tab[lo + li][c] = qr[(size_t)(l0 + lo + li) * lstride + c];
          }
          __syncthreads();
#pragma unroll
          for (int k = 0; k < SRW_ITEMS; k++) {
            const uint32_t t = tok[tid + k * SRW_THREADS];
            if (t != 0xFFFFFFFFu) {
              const CodeT* row = codes + (size_t)t * p.code_stride + l0;
              float sum = cs[k];
              if (vec16) {
                uint32_t ww[SRW_LB / 2];
#pragma unroll
                for (int v = 0; v < SRW_LB / 8; v++) {
                  const uint4 w = __ldg(reinterpret_cast<const uint4*>(row) + v);
                  ww[4 * v] = w.x; ww[4 * v + 1] = w.y; ww[4 * v + 2] = w.z; ww[4 * v + 3] = w.w;
                }
#pragma unroll
                for (int li = 0; li < SRW_LB; li++) {                         // fp32 sum, ascending layer order (+0 for a skipped code)
                  const int c = (int)(short)((ww[li >> 1] >> ((li & 1) * 16)) & 0xFFFFu);
                  if (li >= lo && li < hi && c >= 0 && c < K) sum += __half2float(tab[li][c]);
                }
              } else {
                for (int li = lo; li < hi; li++) {
                  const long long c = (long long)row[li];
                  if (c >= 0 && c < K) sum += __half2float(tab[li][c]);
                }
              }
              cs[k] = sum;
            }
          }
        }
#pragma unroll
        for (int k = 0; k < SRW_ITEMS; k++) {
          const __half h = __float2half_rn(cs[k]);                            // sum(dim=-1) of an fp16 tensor
          rng[k] = (c0 == a) ? h : __float2half_rn(__half2float(rng[k]) + __half2float(h));   // intensities += chunk (fp16)
          cs[k] = 0.f;
        }
      }
#pragma unroll
      for (int k = 0; k < SRW_ITEMS; k++)
        acc[k] = (r == 0) ? rng[k] : __float2half_rn(__half2float(acc[k]) + __half2float(rng[k]));   // accumulation += range (fp16)
      a = b;
    }
#pragma unroll
    for (int k = 0; k < SRW_ITEMS; k++) {
      const long long it = base + tid + (long long)k * SRW_THREADS;
      if (it < per) out[it] = (tok[tid + k * SRW_THREADS] != 0xFFFFFFFFu) ? acc[k] : __float2half(0.f);
    }
    __syncthreads();                                                          // tok is rewritten by the next pass
  }
}

}  // namespace rq
