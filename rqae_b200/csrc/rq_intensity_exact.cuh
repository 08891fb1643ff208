// Bit-exact feature intensities (sm_100a): RQAEFeature.intensity (reference harish-kamath/rqae, rqae/feature.py:102-129)
// with the reference's own roundings, for many features at once.  The tensor-core path (rq_intensity.cuh) sums
// fp16-rounded FACTORS in MMA order; this kernel sums fp16-rounded PRODUCTS in layer order, as torch's CPU kernels do
// for the reference (oracle/feature_oracle.py: intensity_steps).  For feature f, token t and every cut layer:
//
//     p_l   = fp16( w_l * sims[center_f[l]][code_t[l]] )      one rounding (the fp32 product of two fp16 values is exact)
//     run   = +0.0f;  run  = run  + float(p_l),  l = 0, 1, ...  fp32, ascending layers, from +0 (torch's CPU cumsum)
//     wrun  = +0.0f;  wrun = wrun + float(w_l)                 the same for the weights
//     out[f][cut][t] = fp16( float(fp16(run)) / float(fp16(wrun)) )   IEEE fp32 divide (__fdiv_rn), no reciprocal
//
// The running sum starts at +0.0, not at the first product: a leading -0 product (the round_fsq table holds -0
// entries) then gives +0, as in the reference.
//
// Code indexing is the reference's `sims[center, codes]` (torch advanced indexing), for token and center codes alike:
// a code in [-K, 0) reads row / column code + K.  A code outside [-K, K) makes the reference raise; the kernel cannot,
// so such a code contributes a +0 product (the zero row K of the product slab).  The GEMM path differs on negative
// codes: there every code outside [0, K) contributes 0.
//
// Structure.  The K x K table (781 KB at K = 625) does not fit in shared memory; the PRODUCT rows of 8 features over a
// chunk of 8 layers do: P[j][c][g] = fp16(w_{l0+j} * sims[center_g[l0+j]][c]), interleaved by feature, so that one
// 16-byte shared load returns the 8 features' products for one (layer, token code).  A CTA of 256 threads owns a unit
// = (tile of 2048 tokens, group of 8 features); a thread owns 8 tokens and holds their 64 fp32 sums.  Per chunk:
//   1. the 64 center rows and 8 weights of the chunk go to shared memory;
//   2. the CTA writes the chunk's product slab (8 x (K + 1) rows of 16 B) from the table in L2, a thread taking one
//      code and 4 layers per step (32 table loads in flight);
//   3. every thread walks the chunk's layers: per (token, layer) one 16-byte shared load, then per feature one
//      fp16 -> fp32 conversion and one FADD; at a cut layer the 64 quotients are written.  A thread's token codes
//      come as slab byte offsets, two layers per register, loaded one layer pair ahead.
// Two CTAs share an SM (80 KB of slab each, <= 128 registers a thread), so one CTA's staging overlaps the other's sums.
// CTAs are persistent and take units token-tile-major: the CTAs running at one time share a few tiles of codes, which
// stay in L2, while each walks a different feature group.  Every output is one fixed sequential sum, so results do not
// depend on the tiling, the SM count or the stream.
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

namespace rq {

constexpr int IX_THREADS = 256;
constexpr int IX_TPT = 8;                          // tokens per thread
constexpr int IX_TILE = IX_THREADS * IX_TPT;       // 2048 tokens per unit
constexpr int IX_FG = 8;                           // features per unit: one 16-byte row of fp16 products
constexpr int IX_LC = 8;                           // layers per staged chunk
constexpr int IX_ROWS = 640;                       // slab rows per layer: K + 1 <= 640 (row K = the zero row)
constexpr int IX_SLAB = IX_ROWS * 16;              // bytes per layer of the product slab
constexpr int IX_SMEM = IX_LC * IX_SLAB;           // 80 KB dynamic shared memory
constexpr int IX_MAX_LAYERS = 4096;                // deepest cut + 1 (the cut mask's bits)

struct IxParams {
  const __half* sims;          // [K][K] fp16, codebook_sims
  const void* codes;           // [n_tokens][code_stride] of CT
  long long code_stride, n_tokens, n_tiles;
  const int* centers;          // [F][center_stride] int32
  long long center_stride;
  const __half* w;             // [>= L] fp16 layer weights
  __half* out;                 // [F][n_cuts][out_stride]
  long long out_stride;
  int K, F, n_groups, n_cuts, L;                   // L = deepest cut + 1
  unsigned int cut_mask[IX_MAX_LAYERS / 32];       // bit l set: layer l is a cut (ascending bit order = cut order)
};

// Row of `sims` that torch's advanced indexing reads for code c; K (the zero row) where the reference would raise.
__device__ __forceinline__ int ix_row(long long c, int K) {
  if (c < 0) c += K;
  return (c >= 0 && c < K) ? (int)c : K;
}

// The same as a byte offset into a layer's slab, in 32-bit arithmetic where the code type allows.
template <typename CT>
__device__ __forceinline__ uint32_t ix_off(CT c, int K) {
  if constexpr (sizeof(CT) < 8) {
    int v = (int)c;
    v += v < 0 ? K : 0;
    return (uint32_t)((uint32_t)v < (uint32_t)K ? v : K) * 16u;
  } else {
    return (uint32_t)ix_row((long long)c, K) * 16u;
  }
}

template <typename CT>
__global__ void __launch_bounds__(IX_THREADS, 2) rq_intensity_exact_kernel(const IxParams p) {
  extern __shared__ __align__(16) unsigned char ix_smem[];       // [IX_LC][IX_ROWS] rows of 8 fp16 products
  __shared__ int s_crow[IX_LC][IX_FG];                          // center row of every (layer, feature) of the chunk
  __shared__ __half s_w[IX_LC];
  const int tid = threadIdx.x, K = p.K, KR = K + 1;
  const CT* codes = (const CT*)p.codes;
  const long long units = p.n_tiles * p.n_groups;
  const long long cstep = (long long)IX_THREADS * p.code_stride;   // from one of a thread's tokens to the next
  long long t0 = 0;
  const CT* cbase = codes;     // row of the thread's first token
  uint32_t valid = 0;          // bit i: token i of the thread exists
  // codes of layers l0 + j, l0 + j + 1 of this thread's tokens, as byte offsets into a layer's slab (< 2^16), packed
  auto load_pair = [&](int l0, int nl, int j, uint32_t (&o)[IX_TPT]) {
#pragma unroll
    for (int i = 0; i < IX_TPT; i++) {
      uint32_t lo = (uint32_t)K * 16u, hi = lo;
      if ((valid >> i) & 1u) {
        const CT* row = cbase + i * cstep + l0 + j;
        lo = ix_off(__ldg(row), K);
        if (j + 1 < nl) hi = ix_off(__ldg(row + 1), K);
      }
      o[i] = lo | (hi << 16);
    }
  };
  for (long long u = blockIdx.x; u < units; u += gridDim.x) {
    const long long tile = u / p.n_groups;
    const int f0 = (int)(u % p.n_groups) * IX_FG;
    t0 = tile * IX_TILE + tid;                                  // token i of this thread: t0 + i * IX_THREADS
    cbase = codes + t0 * p.code_stride;
    valid = 0;
#pragma unroll
    for (int i = 0; i < IX_TPT; i++) valid |= (t0 + (long long)i * IX_THREADS < p.n_tokens ? 1u : 0u) << i;
    float acc[IX_TPT][IX_FG];
#pragma unroll
    for (int i = 0; i < IX_TPT; i++)
#pragma unroll
      for (int g = 0; g < IX_FG; g++) acc[i][g] = 0.0f;         // +0: a leading -0 product gives +0
    float wrun = 0.0f;
    int cut = 0;
    for (int l0 = 0; l0 < p.L; l0 += IX_LC) {
      const int nl = min(IX_LC, p.L - l0);
      // 1. center rows and weights of the chunk
      if (tid < IX_LC * IX_FG) {
        const int j = tid / IX_FG, g = tid % IX_FG, f = f0 + g;
        s_crow[j][g] = (j < nl && f < p.F) ? ix_row(p.centers[(long long)f * p.center_stride + l0 + j], K) : K;
      } else if (tid < IX_LC * IX_FG + IX_LC) {
        const int j = tid - IX_LC * IX_FG;
        s_w[j] = j < nl ? p.w[l0 + j] : __float2half_rn(0.0f);
      }
      __syncthreads();
      // 2a. this thread's token codes of the chunk's first two layers (the sums load each next pair ahead)
      uint32_t nxt[IX_TPT];
      load_pair(l0, nl, 0, nxt);
      // 2b. product slab: P[j][c][g] = fp16(w_j * sims[crow_g][c]); row K and invalid centers read +0.  A thread
      //     takes one code c and 4 layers per step, so that 32 independent table loads are in flight
      for (int e = tid; e < 2 * IX_THREADS * ((KR + IX_THREADS - 1) / IX_THREADS); e += IX_THREADS) {
        const int c = (e / (2 * IX_THREADS)) * IX_THREADS + e % IX_THREADS, j0 = ((e / IX_THREADS) & 1) * 4;
        if (c >= KR || j0 >= nl) continue;
        __half s[4][IX_FG];
#pragma unroll
        for (int jj = 0; jj < 4; jj++)
#pragma unroll
          for (int g = 0; g < IX_FG; g++) {
            const int r = s_crow[j0 + jj][g];      // K for layers >= nl
            s[jj][g] = (r < K && c < K) ? p.sims[(long long)r * K + c] : __float2half_rn(0.0f);
          }
#pragma unroll
        for (int jj = 0; jj < 4; jj++) {
          const float wj = __half2float(s_w[j0 + jj]);
          __align__(16) __half h[IX_FG];
#pragma unroll
          for (int g = 0; g < IX_FG; g++) h[g] = __float2half_rn(__fmul_rn(wj, __half2float(s[jj][g])));   // exact product, one rounding
          if (j0 + jj < nl) *reinterpret_cast<uint4*>(ix_smem + (j0 + jj) * IX_SLAB + c * 16) = *reinterpret_cast<const uint4*>(h);
        }
      }
      __syncthreads();
      // 3. the sums, layer by layer
      // (one copy of the loop body: unrolled, the cut epilogue's 64 divide sequences would be repeated per layer)
      uint32_t cur[IX_TPT];
#pragma unroll 1
      for (int j = 0; j < nl; j++) {
        if ((j & 1) == 0) {
#pragma unroll
          for (int i = 0; i < IX_TPT; i++) cur[i] = nxt[i];
          if (j + 2 < nl) load_pair(l0, nl, j + 2, nxt);
        }
        const unsigned char* slab = ix_smem + j * IX_SLAB;
        const int sh = (j & 1) * 16;
#pragma unroll
        for (int i = 0; i < IX_TPT; i++) {
          const uint32_t off = (cur[i] >> sh) & 0xFFFFu;
          const uint4 v = *reinterpret_cast<const uint4*>(slab + off);
          const uint32_t pw[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int k = 0; k < 4; k++) {
            const __half2 h2 = *reinterpret_cast<const __half2*>(&pw[k]);
            acc[i][2 * k] = __fadd_rn(acc[i][2 * k], __low2float(h2));
            acc[i][2 * k + 1] = __fadd_rn(acc[i][2 * k + 1], __high2float(h2));
          }
        }
        const int l = l0 + j;
        wrun = __fadd_rn(wrun, __half2float(__ldg(p.w + l)));   // not s_w: a faster thread may already rewrite it
        if ((p.cut_mask[l >> 5] >> (l & 31)) & 1u) {
          const float wd = __half2float(__float2half_rn(wrun));
#pragma unroll
          for (int g = 0; g < IX_FG; g++) {
            if (f0 + g < p.F) {
              __half* orow = p.out + ((long long)(f0 + g) * p.n_cuts + cut) * p.out_stride;
#pragma unroll
              for (int i = 0; i < IX_TPT; i++) {
                const long long t = t0 + (long long)i * IX_THREADS;
                if (t < p.n_tokens)
                  orow[t] = __float2half_rn(__fdiv_rn(__half2float(__float2half_rn(acc[i][g])), wd));
              }
            }
          }
          cut++;
        }
      }
      // step 1 of the next chunk rewrites s_crow / s_w, which only steps 1-2 read (before the second barrier); the
      // slab is rewritten after the next chunk's first barrier, which every thread reaches after its sums
    }
  }
}

}  // namespace rq
