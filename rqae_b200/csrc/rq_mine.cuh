// Top / middle / bottom-k selection over rows of fp16 intensities (sm_100a): rq_mine2_kernel, the exact three-pass
// radix select.
//
// Replaces the per-(feature, layer) `torch.argsort(layer_activations, descending=True)` over the whole
// dataset followed by three slices (scripts/3_make_rqae_features.py:116-128, reference harish-kamath/rqae):
//     top    = sorted[:k]      middle = sorted[n//2 - k//2 : n//2 + k//2]      bottom = sorted[-k:]
// fp16 has 65 536 values, so two histogram passes over 8-bit digits locate the value at each window boundary
// rank, and a third pass collects the window members:
//   pass 1  histogram of the high key byte (raw bit pattern; bins are visited in descending-value order later)
//   pass 2  histogram of the low byte inside the bin that holds the median window (lane-private counters, below);
//           the bins that hold the top / bottom boundaries are tails with few members and use per-warp atomics
//   pass 3  collects the members of the three windows
// The total order is (value descending, index ascending; +0 before -0); torch's argsort is unstable, so the
// reference leaves the order among equal values unspecified -- here it is deterministic.  Warp w owns the
// contiguous slice [w, w+1) * ceil(n / M2_WARPS) of the row, which makes "index ascending" among ties a
// warp-local prefix count plus a per-warp base.  One CTA per row; the row stays in L2 between the passes, so
// HBM sees it once.
//
// The histograms avoid a shared-memory atomic per element: those cost about 2 cycles per element and SM whatever
// the addresses (a first version built on them was ALU-bound, ncu: ALU pipe 72 %, DRAM 5.6 %).  Every LANE of
// every warp owns private 8-bit counters, lp[warp][bin][lane]: an update is a plain LDS.U8 / IADD / STS.U8 that
// cannot collide with another lane (one 32-byte row per bin: at most the four lanes of a quad share a bank), and
// the counters of a warp are folded into 32-bit per-warp totals with DP4A once per 256 elements per lane (an
// 8-bit counter that wrapped is detected by its owner: after a block the counter of the lane's last element must
// be non-zero).
//
// rq_mine3_kernel (rq_mine3.cuh) is the default selection for rows of 16 384 .. 262 144 values; this kernel
// finishes the rows it cannot (list mode) and selects rows of any other length.  RQAE_MINE_V2=1, read per call,
// makes rqae_select_top_middle_bottom_f16 run this kernel for every row, so that the two can be timed and
// compared in one process; it is the library's only selection switch.
#pragma once
#include <cuda_fp16.h>

#include "rq_common.cuh"

namespace rq {

constexpr int MN_KMAX = 256;      // largest window

struct MineParams {
  const __half* vals;     // [rows][row_stride], rows 16-byte aligned, readable up to n rounded up to 8
  long long rows, row_stride, n;
  int k;                  // top_k; the middle window holds 2 * (k / 2) values
  int* idx_out;           // [rows][3][k]   (top, middle, bottom), -1 in unused middle slots
  __half* val_out;        // [rows][3][k]   nullable
  // list mode (rq_mine2_kernel as the fallback of rq_mine3_kernel): the rows to process are row_list[0 .. *row_count)
  const int* row_list = nullptr;
  const int* row_count = nullptr;
  // rq_mine3_kernel: rows it cannot finish are appended to fb_list (counter fb_count) for the list-mode launch
  int* fb_list = nullptr;
  int* fb_count = nullptr;
  int sample_log2 = 4;    // one 32-byte sector out of 2^sample_log2 is sampled
  int c_top = 24;         // sample count that brackets the top / bottom window
  int c_hi = 0, c_lo = 0; // sample ranks that bracket the middle window
};

// key that sorts ascending when the value sorts descending (+0 just before -0)
__device__ __forceinline__ uint32_t mn_dkey(uint32_t u) { return (u & 0x8000u) ? u : (~u & 0x7FFFu); }
__device__ __forceinline__ uint32_t mn_bits(uint32_t d) { return (d & 0x8000u) ? d : (~d & 0x7FFFu); }

#ifndef RQ_M2_WARPS
#define RQ_M2_WARPS 8   /* 8: two CTAs per SM (one row's serial steps run under the other's streaming); 16: one CTA per SM */
#endif
constexpr int M2_WARPS = RQ_M2_WARPS;
constexpr int M2_THREADS = 32 * M2_WARPS;
constexpr int M2_BLOCK_IT = 32;   // 8-element vectors per lane between two folds: 256 elements, see above

constexpr int M2_LP_BYTES = M2_WARPS * 256 * 32;   // lane-private 8-bit counters lp[warp][bin][lane], 8 KB-aligned
constexpr int M2_SMEM_BYTES_PAD = 8192;

struct Mine2Smem {
  uint32_t wtot[M2_WARPS][256];          // per-warp totals (pass 1: high byte; pass 2: low byte inside the dense bin)
  uint32_t ah[3][M2_WARPS][256];         // pass 2: low-byte counts of the other boundary bins (atomics)
  uint32_t pre[257];                     // exclusive prefix over the high-byte bins in descending-value order
  uint32_t scan[M2_WARPS];
  uint32_t bin[4], rem[4], key[4], less[4], slot[4];
  uint32_t base[4][M2_WARPS];
  uint32_t cnt[3];
  uint32_t special, simple, thr[3];      // row flags and the packed-compare thresholds of the pass-2 shortcut
  uint32_t bufk[3][MN_KMAX];
  uint32_t bufi[3][MN_KMAX];
  unsigned char lut[256];                // raw high byte -> 0: not a boundary bin, 1: the dense bin, 2..4: ah[slot - 2]
};

__device__ __forceinline__ void m2_bump(uint32_t addr) {   // lane-private: no other thread touches this byte
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
  asm volatile("st.shared.u8 [%0], %1;" ::"r"(addr), "r"(v + 1u));   // ordered against the other volatile accesses only:
}                                                                   // the folds sit behind __syncwarp / __syncthreads
// two counters of the same lane at once: both loads are in flight together (one trip through shared memory for
// two values); if they are the SAME counter the second store carries both increments
__device__ __forceinline__ void m2_bump2(uint32_t a0, uint32_t a1) {
  uint32_t v0, v1;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v0) : "r"(a0));
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v1) : "r"(a1));
  asm volatile("st.shared.u8 [%0], %1;" ::"r"(a0), "r"(v0 + 1u));
  asm volatile("st.shared.u8 [%0], %1;" ::"r"(a1), "r"(v1 + 1u + (a0 == a1 ? 1u : 0u)));
}
__device__ __forceinline__ uint32_t m2_peek(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}

// fold the warp's lane-private counters into wtot[warp][*] and clear them (whole warp, converged)
__device__ __forceinline__ void m2_fold(Mine2Smem& sm, unsigned char* lp, int warp, int lane) {
  __syncwarp();
  const uint4* rows = reinterpret_cast<const uint4*>(lp + warp * 8192);
  uint4* rows_w = reinterpret_cast<uint4*>(lp + warp * 8192);
#pragma unroll 4
  for (int m = 0; m < 16; m++) {
    // lane -> (bin 16 m + lane / 2, half lane % 2): a warp load covers 512 contiguous bytes
    const uint4 v = rows[m * 32 + lane];
    uint32_t sum = __dp4a(v.x, 0x01010101u, 0u);
    sum = __dp4a(v.y, 0x01010101u, sum);
    sum = __dp4a(v.z, 0x01010101u, sum);
    sum = __dp4a(v.w, 0x01010101u, sum);
    sum += __shfl_xor_sync(0xffffffffu, sum, 1);
    if ((lane & 1) == 0 && sum != 0) sm.wtot[warp][16 * m + (lane >> 1)] += sum;
    rows_w[m * 32 + lane] = make_uint4(0u, 0u, 0u, 0u);
  }
  __syncwarp();
}

__global__ void __launch_bounds__(M2_THREADS, 16 / M2_WARPS) rq_mine2_kernel(const MineParams p) {
  extern __shared__ __align__(16) unsigned char m2_raw[];
  // the counters sit on an 8 KB boundary so that the address of a counter is (bin << 5) OR-ed into the lane's base
  const uint32_t raw32 = smem_u32(m2_raw);
  const uint32_t lp32 = (raw32 + 8191u) & ~8191u;
  unsigned char* const lp = m2_raw + (lp32 - raw32);
  Mine2Smem& sm = *reinterpret_cast<Mine2Smem*>(lp + M2_LP_BYTES);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long n = p.n;
  const int k = p.k, kh = k / 2;
  const long long seg = ((n + M2_WARPS - 1) / M2_WARPS + 7) / 8 * 8;     // per-warp slice, multiple of 8
  const long long w_lo = warp * seg, w_hi = (w_lo + seg < n) ? w_lo + seg : n;
  const long long m0 = n / 2 - kh, m1 = n / 2 + kh;
  const long long rank[4] = {(long long)k - 1, m0, m1 - 1, n - k};
  const uint32_t my = lp32 + (uint32_t)warp * 8192u + (uint32_t)lane;   // bits 5..12 are free for the bin

  {   // the lane-private counters start cleared and every fold leaves them cleared
    uint4* z = reinterpret_cast<uint4*>(lp);
    for (int i = tid; i < M2_LP_BYTES / 16; i += M2_THREADS) z[i] = make_uint4(0u, 0u, 0u, 0u);
  }

  const long long n_rows = p.row_count ? (long long)*p.row_count : p.rows;
  for (long long ri = blockIdx.x; ri < n_rows; ri += gridDim.x) {
    const long long row = p.row_list ? (long long)p.row_list[ri] : ri;
    const uint4* src = reinterpret_cast<const uint4*>(p.vals + row * p.row_stride);
    for (int i = tid; i < M2_WARPS * 256; i += M2_THREADS) (&sm.wtot[0][0])[i] = 0;
    for (int i = tid; i < 3 * M2_WARPS * 256; i += M2_THREADS) (&sm.ah[0][0][0])[i] = 0;
    if (tid < 3) sm.cnt[tid] = 0;
    if (tid < 256) sm.lut[tid] = 0;
    if (tid == 3) sm.special = 0;
    __syncthreads();

    // ---- pass 1: high byte ----
    for (long long ib = w_lo; ib < w_hi; ib += 256LL * M2_BLOCK_IT) {
      uint32_t last = 0;
      // two vectors per step, and the next step's two loads are issued before this step's updates (the update chain
      // of a step is about as long as a trip to L2 / HBM)
      uint4 na = make_uint4(0u, 0u, 0u, 0u), nb = na;
      {
        const long long j0 = ib + lane * 8, j1 = j0 + 256;
        if (j0 < w_hi) na = __ldg(src + j0 / 8);
        if (j1 < w_hi) nb = __ldg(src + j1 / 8);
      }
      for (int b = 0; b < M2_BLOCK_IT; b += 2) {
        const long long i0 = ib + (long long)b * 256 + lane * 8, i1 = i0 + 256;
        if (i0 >= w_hi) break;
        const bool two = i1 < w_hi;
        const uint4 va = na, vb = nb;
        if (b + 2 < M2_BLOCK_IT) {
          const long long j0 = i0 + 512, j1 = i0 + 768;
          if (j0 < w_hi) na = __ldg(src + j0 / 8);
          if (j1 < w_hi) nb = __ldg(src + j1 / 8);
        }
        const uint32_t w8[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
        if (two && i1 + 8 <= w_hi) {
#pragma unroll
          for (int e = 0; e < 8; e++) {
            last = ((w8[e] >> 19) & 0x1FE0u) | my;
            m2_bump2(((w8[e] >> 3) & 0x1FE0u) | my, last);       // ((bits >> 8) & 0xFF) * 32
          }
        } else {
#pragma unroll
          for (int e = 0; e < 16; e++) {
            const long long pos = (e < 8 ? i0 + e : i1 + (e - 8));
            if ((e < 8 || two) && pos < w_hi) {
              last = ((((w8[e >> 1] >> ((e & 1) * 16)) >> 8) & 0xFFu) << 5) | my;
              m2_bump(last);
            }
          }
        }
      }
      if (last != 0 && m2_peek(last) == 0) atomicAdd(&sm.wtot[warp][(last >> 5) & 0xFFu], 256u);   // the counter wrapped
      m2_fold(sm, lp, warp, lane);
    }
    __syncthreads();
    // bin totals in descending-value order (positive patterns from the top down, then negative ones upwards) and
    // their exclusive prefix
    {
      uint32_t c = 0;
      if (tid < 256) {
        const int raw = (tid & 0x80) ? tid : (~tid & 0x7F);
#pragma unroll
        for (int w = 0; w < M2_WARPS; w++) c += sm.wtot[w][raw];
        // inf / NaN patterns (exponent 31) anywhere in the row: the packed-compare shortcuts of passes 2 and 3 are off
        if ((raw & 0x7C) == 0x7C && c != 0) sm.special = 1;
      }
      uint32_t x = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
      }
      if (lane == 31) sm.scan[warp] = x;
      __syncthreads();
      if (warp == 0) {
        uint32_t t = lane < M2_WARPS ? sm.scan[lane] : 0u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t y = __shfl_up_sync(0xffffffffu, t, o);
          if (lane >= o) t += y;
        }
        if (lane < M2_WARPS) sm.scan[lane] = t;
      }
      __syncthreads();
      if (tid < 256) sm.pre[tid] = x - c + (warp > 0 ? sm.scan[warp - 1] : 0u);
      if (tid == 0) sm.pre[256] = (uint32_t)n;
    }
    __syncthreads();
    for (int i = tid; i < M2_WARPS * 256; i += M2_THREADS) (&sm.wtot[0][0])[i] = 0;   // reused by pass 2
    if (tid < 4) {   // last bin whose exclusive prefix is <= rank
      const uint32_t r = (uint32_t)rank[tid];
      int lo = 0, hi = 255;
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (sm.pre[mid] <= r) lo = mid; else hi = mid - 1;
      }
      sm.bin[tid] = lo;
      sm.rem[tid] = r - sm.pre[lo];
    }
    __syncthreads();
    if (tid == 0) {   // the median's bin is counted lane-privately, every other distinct boundary bin with atomics
      int next = 2;
      const int order[4] = {1, 2, 0, 3};
      for (int q = 0; q < 4; q++) {
        const int j = order[q];
        int s = 0;
        for (int q2 = 0; q2 < q; q2++)
          if (sm.bin[order[q2]] == sm.bin[j]) s = (int)sm.slot[order[q2]];
        if (s == 0) s = (q == 0) ? 1 : next++;
        sm.slot[j] = (uint32_t)s;
        const int d = (int)sm.bin[j];
        sm.lut[(d & 0x80) ? d : (~d & 0x7F)] = (unsigned char)s;
      }
      // Shortcut of pass 2: besides the dense bin only TAIL bins are boundary bins (both median ranks in one bin) and
      // the row holds no inf / NaN.  A value can then only belong to a tail bin if it is >= the smallest value of the
      // top boundary bin or <= the largest value of the bottom one -- one packed fp16 compare per pair of values.
      sm.simple = (sm.special == 0 && sm.slot[2] == 1) ? 1u : 0u;
      const int d0 = (int)sm.bin[0], d3 = (int)sm.bin[3];
      const uint32_t r0 = (d0 & 0x80) ? d0 : (~d0 & 0x7F), r3 = (d3 & 0x80) ? d3 : (~d3 & 0x7F);
      // bit patterns of the smallest value of bin r0 / the largest value of bin r3 (negative: larger pattern = smaller value)
      const uint32_t lo0 = (r0 & 0x80) ? ((r0 << 8) | 0xFFu) : (r0 << 8);
      const uint32_t hi3 = (r3 & 0x80) ? (r3 << 8) : ((r3 << 8) | 0xFFu);
      sm.thr[0] = sm.slot[0] == 1 ? 0x7C00u : lo0;    // +inf: never reached in a simple row
      sm.thr[1] = sm.slot[3] == 1 ? 0xFC00u : hi3;    // -inf
      const int dd = (int)sm.bin[1];
      sm.thr[2] = (dd & 0x80) ? dd : (~dd & 0x7F);   // raw high byte of the dense bin
    }
    __syncthreads();

    // ---- pass 2: low byte inside the boundary bins ----
    const bool simple = sm.simple != 0;
    for (long long ib = w_lo; ib < w_hi; ib += 256LL * M2_BLOCK_IT) {
      uint32_t last = 0;
      if (simple) {
        const uint32_t dlo = sm.thr[2] << 8, dhi = sm.thr[2] << 24;
        const uint32_t ttop = sm.thr[0] * 0x10001u, tbot = sm.thr[1] * 0x10001u;
        const __half2 htop = *reinterpret_cast<const __half2*>(&ttop), hbot = *reinterpret_cast<const __half2*>(&tbot);
        uint4 nv = make_uint4(0u, 0u, 0u, 0u);
        if (ib + lane * 8 < w_hi) nv = __ldg(src + (ib + lane * 8) / 8);
        for (int b = 0; b < M2_BLOCK_IT; b++) {
          const long long i0 = ib + (long long)b * 256 + lane * 8;
          if (i0 >= w_hi) break;
          const uint4 v = nv;
          if (b + 1 < M2_BLOCK_IT && i0 + 256 < w_hi) nv = __ldg(src + (i0 + 256) / 8);
          const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
          if (i0 + 8 <= w_hi) {
#pragma unroll
            for (int e = 0; e < 4; e++) {
              const uint32_t w = w4[e];
              const __half2 h = *reinterpret_cast<const __half2*>(&w);
              const uint32_t tm = __hge2_mask(h, htop) | __hle2_mask(h, hbot);
              if ((w & 0xFF00u) == dlo) { last = ((w << 5) & 0x1FE0u) | my; m2_bump(last); }
              if ((w & 0xFF000000u) == dhi) { last = ((w >> 11) & 0x1FE0u) | my; m2_bump(last); }
              if (tm != 0) {   // a value in (or beyond) a tail boundary bin: a few hundred per row
                if (tm & 0xFFFFu) {
                  const uint32_t s = sm.lut[(w >> 8) & 0xFFu];
                  if (s >= 2) atomicAdd(&sm.ah[s - 2][warp][w & 0xFFu], 1u);
                }
                if (tm >> 16) {
                  const uint32_t s = sm.lut[w >> 24];
                  if (s >= 2) atomicAdd(&sm.ah[s - 2][warp][(w >> 16) & 0xFFu], 1u);
                }
              }
            }
          } else {
#pragma unroll
            for (int e = 0; e < 8; e++) {
              if (i0 + e < w_hi) {
                const uint32_t u = (w4[e >> 1] >> ((e & 1) * 16)) & 0xFFFFu;
                const uint32_t s = sm.lut[u >> 8];
                if (s == 1) { last = ((u & 0xFFu) << 5) | my; m2_bump(last); }
                else if (s != 0) atomicAdd(&sm.ah[s - 2][warp][u & 0xFFu], 1u);
              }
            }
          }
        }
      } else {
        for (int b = 0; b < M2_BLOCK_IT; b++) {
          const long long i0 = ib + (long long)b * 256 + lane * 8;
          if (i0 >= w_hi) break;
          const uint4 v = __ldg(src + i0 / 8);
          const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
          const bool full = i0 + 8 <= w_hi;
          uint32_t sl[8];
#pragma unroll
          for (int e = 0; e < 8; e++) sl[e] = sm.lut[((w4[e >> 1] >> ((e & 1) * 16)) >> 8) & 0xFFu];
#pragma unroll
          for (int e = 0; e < 8; e++) {
            if (full || i0 + e < w_hi) {
              const uint32_t u = (w4[e >> 1] >> ((e & 1) * 16)) & 0xFFFFu;
              if (sl[e] == 1) { last = ((u & 0xFFu) << 5) | my; m2_bump(last); }
              else if (sl[e] != 0) atomicAdd(&sm.ah[sl[e] - 2][warp][u & 0xFFu], 1u);
            }
          }
        }
      }
      if (last != 0 && m2_peek(last) == 0) atomicAdd(&sm.wtot[warp][(last >> 5) & 0xFFu], 256u);
      m2_fold(sm, lp, warp, lane);
    }
    __syncthreads();
    if (warp < 4) {   // warp j resolves boundary j: lane owns 8 consecutive low-byte values in descending-value order
      const int j = warp;
      const uint32_t dbin = sm.bin[j];
      const bool positive = (dbin & 0x80u) == 0;
      const uint32_t(*cs)[256] = sm.slot[j] == 1 ? sm.wtot : sm.ah[sm.slot[j] - 2];
      uint32_t c[8], tot = 0;
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int d = lane * 8 + i, raw = positive ? 255 - d : d;
        uint32_t a = 0;
#pragma unroll
        for (int w = 0; w < M2_WARPS; w++) a += cs[w][raw];
        c[i] = a;
        tot += a;
      }
      uint32_t incl = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += y;
      }
      const uint32_t rem = sm.rem[j];
      const bool mine = rem >= incl - tot && rem < incl;      // exactly one lane
      int sb = 0;
      if (mine) {
        uint32_t run = incl - tot;
#pragma unroll
        for (int i = 0; i < 8; i++) {
          if (rem >= run && rem < run + c[i]) {
            sb = lane * 8 + i;
            sm.key[j] = (dbin << 8) | (uint32_t)sb;
            sm.less[j] = sm.pre[dbin] + run;
          }
          run += c[i];
        }
      }
      const uint32_t sel = __ballot_sync(0xffffffffu, mine);
      sb = __shfl_sync(0xffffffffu, sb, __ffs(sel) - 1);
      // tie base of warp `lane`: ties at the boundary key in the warps before it
      const uint32_t t = lane < M2_WARPS ? cs[lane][positive ? 255 - sb : sb] : 0u;
      uint32_t ti = t;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, ti, o);
        if (lane >= o) ti += y;
      }
      if (lane < M2_WARPS) sm.base[j][lane] = ti - t;
    }
    __syncthreads();

    // ---- pass 3: collect the members of the three windows ----
    {
      const uint32_t K0 = sm.key[0], K1 = sm.key[1], K2 = sm.key[2], K3 = sm.key[3];
      const uint32_t top_take = (uint32_t)k - sm.less[0];                    // tie ranks < top_take are in top
      const uint32_t mid_skip = (uint32_t)m0 - sm.less[1];                   // tie ranks >= mid_skip are in middle
      const uint32_t mid_take = (uint32_t)m1 - sm.less[2];                   // tie ranks < mid_take are in middle
      const uint32_t bot_skip = (uint32_t)(n - k) - sm.less[3];              // tie ranks >= bot_skip are in bottom
      uint32_t tc[4] = {sm.base[0][warp], sm.base[1][warp], sm.base[2][warp], sm.base[3][warp]};
      // Rows without inf / NaN: a value is a candidate only if it is >= value(K0), <= value(K3) or inside
      // [value(K2), value(K1)] -- packed fp16 compares (a superset where +0 / -0 are concerned; the exact key test
      // follows for the values that pass).
      const bool quick = sm.special == 0;
      const uint32_t b0 = mn_bits(K0) * 0x10001u, b1 = mn_bits(K1) * 0x10001u, b2 = mn_bits(K2) * 0x10001u, b3 = mn_bits(K3) * 0x10001u;
      const __half2 h0 = *reinterpret_cast<const __half2*>(&b0), h1 = *reinterpret_cast<const __half2*>(&b1);
      const __half2 h2 = *reinterpret_cast<const __half2*>(&b2), h3 = *reinterpret_cast<const __half2*>(&b3);
      auto append = [&](int wdw, uint32_t dd, uint32_t index) {
        const uint32_t s = atomicAdd(&sm.cnt[wdw], 1u);
        if (s < MN_KMAX) { sm.bufk[wdw][s] = dd; sm.bufi[wdw][s] = index; }
      };
      uint4 nv = make_uint4(0u, 0u, 0u, 0u);
      if (w_lo + lane * 8 < w_hi) nv = __ldg(src + (w_lo + lane * 8) / 8);
      for (long long i0 = w_lo + lane * 8; i0 - lane * 8 < w_hi; i0 += 256) {   // whole warp iterates together
        const uint4 v = nv;
        nv = make_uint4(0u, 0u, 0u, 0u);
        if (i0 + 256 < w_hi) nv = __ldg(src + (i0 + 256) / 8);   // the next vector is in flight while this one is examined
        const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
        // per pair of values: which halves can be candidates at all
        uint32_t qm[4] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
        if (quick) {
#pragma unroll
          for (int e = 0; e < 4; e++) {
            const __half2 h = *reinterpret_cast<const __half2*>(&w4[e]);
            qm[e] = __hge2_mask(h, h0) | __hle2_mask(h, h3) | (__hle2_mask(h, h1) & __hge2_mask(h, h2));
          }
        }
        const bool lane_any = i0 < w_hi && (qm[0] | qm[1] | qm[2] | qm[3]) != 0;
        if (!__any_sync(0xffffffffu, lane_any)) continue;
        // Values strictly inside a window are appended at once; values EQUAL to a boundary key are ties whose
        // membership depends on their rank among the equal values (index order): counted here, ranked below.
        uint32_t neq[4] = {0, 0, 0, 0};
        if (lane_any) {
#pragma unroll
          for (int e = 0; e < 8; e++) {
            if (((qm[e >> 1] >> ((e & 1) * 16)) & 0xFFFFu) != 0 && i0 + e < w_hi) {
              const uint32_t dd = mn_dkey((w4[e >> 1] >> ((e & 1) * 16)) & 0xFFFFu);
              const bool e0 = dd == K0, e1 = dd == K1, e2 = dd == K2, e3 = dd == K3;
              if (e0 | e1 | e2 | e3) {
                neq[0] += e0; neq[1] += e1; neq[2] += e2; neq[3] += e3;
              } else {
                const uint32_t index = (uint32_t)(i0 + e);
                if (dd < K0) append(0, dd, index);
                if (kh > 0 && dd > K1 && dd < K2) append(1, dd, index);
                if (dd > K3) append(2, dd, index);
              }
            }
          }
        }
        const bool lane_tie = (neq[0] | neq[1] | neq[2] | neq[3]) != 0;
        if (!__any_sync(0xffffffffu, lane_tie)) continue;
        uint32_t ex[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
          uint32_t x = neq[j];
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
          }
          ex[j] = tc[j] + x - neq[j];
          tc[j] += __shfl_sync(0xffffffffu, x, 31);
        }
        if (lane_tie) {
#pragma unroll
          for (int e = 0; e < 8; e++) {
            if (i0 + e < w_hi) {
              const uint32_t dd = mn_dkey((w4[e >> 1] >> ((e & 1) * 16)) & 0xFFFFu);
              if (dd == K0 || dd == K1 || dd == K2 || dd == K3) {
                const uint32_t t0 = ex[0], t1 = ex[1], t2 = ex[2], t3 = ex[3];
                ex[0] += dd == K0; ex[1] += dd == K1; ex[2] += dd == K2; ex[3] += dd == K3;
                const bool in_top = dd < K0 || (dd == K0 && t0 < top_take);
                const bool in_mid = kh > 0 && (dd > K1 || (dd == K1 && t1 >= mid_skip)) && (dd < K2 || (dd == K2 && t2 < mid_take));
                const bool in_bot = dd > K3 || (dd == K3 && t3 >= bot_skip);
                const uint32_t index = (uint32_t)(i0 + e);
                if (in_top) append(0, dd, index);
                if (in_mid) append(1, dd, index);
                if (in_bot) append(2, dd, index);
              }
            }
          }
        }
      }
    }
    __syncthreads();

    // ---- order each window by (key, index) and write it out ----
    for (int w = 0; w < 3; w++) {
      const int cnt = min((int)sm.cnt[w], MN_KMAX);
      int* io = p.idx_out + (row * 3 + w) * (long long)k;
      __half* vo = p.val_out ? p.val_out + (row * 3 + w) * (long long)k : nullptr;
      if (tid < cnt) {
        const uint32_t dk = sm.bufk[w][tid], di = sm.bufi[w][tid];
        int r = 0;
        for (int o = 0; o < cnt; o++) {
          const uint32_t ok = sm.bufk[w][o], oi = sm.bufi[w][o];
          r += (ok < dk) || (ok == dk && oi < di);
        }
        if (r < k) {
          io[r] = (int)di;
          if (vo) vo[r] = __ushort_as_half((unsigned short)mn_bits(dk));
        }
      } else if (tid < k) {
        if (tid >= cnt) { io[tid] = -1; if (vo) vo[tid] = __ushort_as_half((unsigned short)0); }
      }
    }
    __syncthreads();
  }
}

}  // namespace rq
