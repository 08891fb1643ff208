// rq_mine3_kernel: top / middle / bottom-k selection (scripts/3_make_rqae_features.py:116-128, reference
// harish-kamath/rqae) with ONE streaming pass over a row instead of three histogram passes.
//
// rq_mine2_kernel is exact but instruction-bound (49 thread-instructions per value over its three passes; an
// HBM-bound pass affords about 11).  Here the four window boundaries are BRACKETED from a 1/16 sample of the row
// before the row is streamed:
//   A  sample   one 32-byte sector out of every 16 (the sector inside a group is picked by a hash, so that a period
//               in the token order cannot alias with the sample); a two-level radix select over the sample yields the
//               keys at four sample ranks: T_top (c_top sample values lie at or above it), T_bot, and [M_lo, M_hi]
//               around the median ranks (4 sigma of the sample's rank error on either side).  Exact sample order
//               statistics, not bin edges: the bracket's size does not depend on the magnitude of the row.
//   B  stream   every value is compared against the thresholds with packed fp16 compares (two values per
//               instruction): values above M_hi are COUNTED (G, dp4a over the compare masks), values >= T_top,
//               <= T_bot or inside [M_lo, M_hi] (about 6 % of a row) are appended, key and position, to the warp's own
//               region of a shared-memory candidate buffer.  Warp w streams the contiguous slice w of the row and
//               appends in index order (slots from two packed warp scans per 2 KB step, no atomics), so the buffer as a
//               whole is in index order.  Bracket members are counted in their level-1 histogram on the way.
//   C  select   exact selection among the candidates, the three windows side by side: a two-level radix select over
//               each class's key range finds the keys at the window's first and last rank; keys strictly between them
//               are members, a key EQUAL to a boundary key is a member according to its rank among the equal values in
//               index order (= equal values in earlier regions + equal values earlier in the region; computed over a
//               short per-warp list of the keys inside the windows' key ranges: tie groups are never sorted); the <= 256 members of a window are ordered by a 64-bit (key, index)
//               rank sort.
// The brackets are VERIFIED, not trusted: G <= m0, G + |bracket| >= m1, at least k values in either tail class, no
// NaN in the row (a NaN becomes a candidate through an unordered compare and is seen in step C), no region overflow.
// A row that fails any of it is appended to a fallback list and finished by rq_mine2_kernel in list mode (same stream,
// no host round trip), so the result is the exact selection in the same total order (value descending, index ascending;
// +0 before -0) whatever the data looks like -- constant rows, rows whose bracket holds more than 768 candidates per
// warp and rows with NaN simply take the old path.  fp compares treat +0 and -0 as equal; both then fall into the same
// class and are told apart by their keys in step C.  16 384 <= n <= 262 144 (the sample statistics and the 18-bit
// position); other sizes go to rq_mine2_kernel directly.
#pragma once
#include <cuda_fp16.h>

#include <type_traits>

#include "rq_mine.cuh"

namespace rq {

constexpr int M3_THREADS = 512;
constexpr int M3_WARPS = M3_THREADS / 32;
constexpr int M3_WCAP = 768;       // candidates per warp and row: every warp appends to its own region (no atomics)
constexpr int M3_CAP = M3_WCAP * M3_WARPS;
constexpr int M3_LIST = MN_KMAX;   // members of one window
constexpr int M3_BINS = 2048;
constexpr int M3_SORT_THREADS = 160;   // threads per class in the rank sort (five warps each)

struct Mine3Smem {
  uint32_t hist[3][M3_BINS];         // [0] also holds the sample histogram of step A
  uint32_t candi[M3_CAP];
  unsigned short candk[M3_CAP];
  unsigned long long lk[3][M3_LIST]; // key << 32 | index of the members of each window
  uint32_t h2[3][2][32];
  uint32_t scan[3][M3_WARPS];
  uint32_t wcount[M3_WARPS];         // candidates of each warp
  uint32_t G, nan, lcount[3];
  uint32_t tbin[4], tex[4], tkey[4]; // level-1 bin, its exclusive prefix and the key of the four thresholds (T_top, T_bot, M_hi, M_lo)
  uint32_t binA[3], exA[3], binB[3], exB[3];   // level-1 bins of a window's first / last rank and their exclusive prefixes
  uint32_t klo[3], khi[3], less_lo[3], less_hi[3];
  uint32_t tie[6][M3_WARPS];         // per warp: candidates equal to klo / khi of each class
};

__device__ __forceinline__ uint32_t m3_hash(uint32_t g, uint32_t row) {
  uint32_t h = g * 0x9E3779B1u + row * 0x85EBCA6Bu + 0x165667B1u;
  h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12; h *= 0x297A2D39u; h ^= h >> 15;
  return h;
}

__device__ __forceinline__ void m3_prefetch_l2(const void* ptr, uint32_t bytes) {   // 16-byte aligned, multiple of 16
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(ptr), "r"(bytes) : "memory");
}
__device__ __forceinline__ int m3_dp4a_su(uint32_t a_signed_bytes, uint32_t b_unsigned_bytes, int c) {
  int d;
  asm("dp4a.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a_signed_bytes), "r"(b_unsigned_bytes), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t m3_sel3(int c, uint32_t a0, uint32_t a1, uint32_t a2) { return c == 0 ? a0 : (c == 1 ? a1 : a2); }

__device__ __forceinline__ uint32_t m3_warp_inclusive(uint32_t v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += y;
  }
  return v;
}

__global__ void __launch_bounds__(M3_THREADS, 2) rq_mine3_kernel(const MineParams p) {
  extern __shared__ __align__(16) unsigned char m3_raw[];
  Mine3Smem& sm = *reinterpret_cast<Mine3Smem*>(m3_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long n = p.n;
  const int k = p.k, kh = k / 2;
  const long long m0 = n / 2 - kh, m1 = n / 2 + kh;
  const long long nv = n / 8;                                // whole 16-byte vectors
  const int slog = p.sample_log2;
  const long long ngroups = (n / 16) >> slog;                // sample: one sector (16 values) per group
  const uint32_t ms = (uint32_t)ngroups * 16u;

  for (long long row = blockIdx.x; row < p.rows; row += gridDim.x) {
    const uint4* src = reinterpret_cast<const uint4*>(p.vals + row * p.row_stride);
    const unsigned short* src16 = reinterpret_cast<const unsigned short*>(p.vals + row * p.row_stride);
    for (int i = tid; i < M3_BINS; i += M3_THREADS) sm.hist[0][i] = 0;
    if (tid < 128) (&sm.h2[0][0][0])[tid] = 0;
    if (tid == 0) {
      sm.G = 0; sm.nan = 0;
      for (int j = 0; j < 4; j++) { sm.tbin[j] = 0; sm.tex[j] = 0; }
    }
    __syncthreads();

    // ---- A: two-level radix select over the sample: the keys at four sample ranks are the thresholds ----
    // 0-based ranks in descending-value order: T_top = rank c_top - 1, T_bot = rank ms - c_top, M_hi = rank c_hi,
    // M_lo = rank c_lo - 1
    const uint32_t rk[4] = {(uint32_t)p.c_top - 1u, ms - (uint32_t)p.c_top, (uint32_t)(p.c_hi > 0 ? p.c_hi : 0),
                            (uint32_t)p.c_lo - 1u < ms ? (uint32_t)p.c_lo - 1u : ms - 1u};
    for (long long g = tid; g < ngroups; g += M3_THREADS) {
      const long long sector = (g << slog) + (m3_hash((uint32_t)g, (uint32_t)row) >> (32 - slog));
      const uint4 a = __ldg(src + sector * 2), b = __ldg(src + sector * 2 + 1);
      const uint32_t w8[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
      for (int e = 0; e < 8; e++) {
        const uint32_t w = w8[e];
        const uint32_t d2 = w ^ ((((w >> 15) & 0x00010001u) * 0x7FFFu) ^ 0x7FFF7FFFu);   // packed descending keys
        atomicAdd(&sm.hist[0][(d2 & 0xFFFFu) >> 5], 1u);
        atomicAdd(&sm.hist[0][d2 >> 21], 1u);
      }
    }
    __syncthreads();
    {
      uint32_t c[4], tot = 0;
#pragma unroll
      for (int i = 0; i < 4; i++) { c[i] = sm.hist[0][tid * 4 + i]; tot += c[i]; }
      const uint32_t inc = m3_warp_inclusive(tot, lane);
      if (lane == 31) sm.scan[0][warp] = inc;
      __syncthreads();
      uint32_t ex = inc - tot;
#pragma unroll
      for (int w = 0; w < M3_WARPS; w++) ex += w < warp ? sm.scan[0][w] : 0u;
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const uint32_t in = ex + c[i];
#pragma unroll
        for (int j = 0; j < 4; j++)
          if (ex <= rk[j] && rk[j] < in) { sm.tbin[j] = (uint32_t)tid * 4 + i; sm.tex[j] = ex; }
        ex = in;
      }
    }
    __syncthreads();
    {   // level 2: the low five key bits inside the four bins (the sample is read again: it sits in L1 / L2)
      const uint32_t b0 = sm.tbin[0], b1 = sm.tbin[1], b2 = sm.tbin[2], b3 = sm.tbin[3];
      for (long long g = tid; g < ngroups; g += M3_THREADS) {
        const long long sector = (g << slog) + (m3_hash((uint32_t)g, (uint32_t)row) >> (32 - slog));
        const uint4 a = __ldg(src + sector * 2), b = __ldg(src + sector * 2 + 1);
        const uint32_t w8[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int e = 0; e < 8; e++) {
          const uint32_t w = w8[e];
          const uint32_t d2 = w ^ ((((w >> 15) & 0x00010001u) * 0x7FFFu) ^ 0x7FFF7FFFu);
#pragma unroll
          for (int hh = 0; hh < 2; hh++) {
            const uint32_t d = hh ? d2 >> 16 : d2 & 0xFFFFu, bin = d >> 5;
            if (bin == b0) atomicAdd(&sm.h2[0][0][d & 31u], 1u);
            if (bin == b1) atomicAdd(&sm.h2[0][1][d & 31u], 1u);
            if (bin == b2) atomicAdd(&sm.h2[1][0][d & 31u], 1u);
            if (bin == b3) atomicAdd(&sm.h2[1][1][d & 31u], 1u);
          }
        }
      }
      __syncthreads();
      if (warp < 4) {
        const uint32_t cnt = (&sm.h2[0][0][0])[warp * 32 + lane];
        const uint32_t inc = m3_warp_inclusive(cnt, lane);
        const uint32_t target = rk[warp] - sm.tex[warp];
        const uint32_t sel = __ballot_sync(0xffffffffu, inc - cnt <= target && target < inc);
        if (lane == 0) sm.tkey[warp] = (sm.tbin[warp] << 5) | (sel ? (uint32_t)__ffs(sel) - 1u : 0u);
      }
      __syncthreads();
    }
    // bit patterns of the thresholds (rank c_hi < 0: the bracket starts at the very top, key 0)
    const uint32_t Ttop = mn_bits(sm.tkey[0]), Tbot = mn_bits(sm.tkey[1]);
    const uint32_t Mhi = mn_bits(p.c_hi >= 0 ? sm.tkey[2] : 0u), Mlo = mn_bits(sm.tkey[3]);
    const uint32_t ttop2 = Ttop * 0x10001u, tbot2 = Tbot * 0x10001u, mhi2 = Mhi * 0x10001u, mlo2 = Mlo * 0x10001u;
    const __half2 htop = *reinterpret_cast<const __half2*>(&ttop2), hbot = *reinterpret_cast<const __half2*>(&tbot2);
    const __half2 hmhi = *reinterpret_cast<const __half2*>(&mhi2), hmlo = *reinterpret_cast<const __half2*>(&mlo2);
    const __half stop = __ushort_as_half((unsigned short)Ttop), sbot = __ushort_as_half((unsigned short)Tbot);
    const __half smhi = __ushort_as_half((unsigned short)Mhi), smlo = __ushort_as_half((unsigned short)Mlo);
    // key ranges [kb, ke] of the three classes (0: values >= T_top, 1: the bracket of the median, 2: values <= T_bot) and
    // the bin widths of their level-1 histograms.  +0 / -0 compare equal: a range that ends at one of them is widened
    // over both.
    const uint32_t kb0 = 0u, kb1 = Mhi == 0x8000u ? 0x7FFFu : mn_dkey(Mhi), kb2 = Tbot == 0x8000u ? 0x7FFFu : mn_dkey(Tbot);
    const uint32_t ke0 = Ttop == 0x0000u ? 0x8000u : mn_dkey(Ttop), ke1 = Mlo == 0x0000u ? 0x8000u : mn_dkey(Mlo), ke2 = 0xFFFFu;
    int sh0 = 0, sh1 = 0, sh2 = 0;
    while (((ke0 - kb0) >> sh0) >= (uint32_t)M3_BINS) sh0++;
    while (((ke1 - kb1) >> sh1) >= (uint32_t)M3_BINS) sh1++;
    while (((ke2 - kb2) >> sh2) >= (uint32_t)M3_BINS) sh2++;
    // zero what steps B and C accumulate into (hist[0] is free again after the barrier above)
    for (int i = tid; i < 3 * M3_BINS; i += M3_THREADS) (&sm.hist[0][0])[i] = 0;
    if (tid < 192) (&sm.h2[0][0][0])[tid] = 0;
    if (tid < 3) sm.lcount[tid] = 0;
    __syncthreads();

    // ---- B: one pass over the row ----
    // A NaN compares "greater or unordered" to T_top, so it becomes a candidate; step C sees its bit pattern and sends
    // the row to the fallback (no separate NaN test per value).
    {
      uint32_t gcount = 0;
      uint32_t gacc = 0;                                              // 510 x (values above the bracket)
      uint32_t wcnt = 0;                                              // candidates of this warp so far (warp-uniform)
      const uint32_t ka = smem_u32(sm.candk) + (uint32_t)warp * (M3_WCAP * 2u);
      const uint32_t ia = smem_u32(sm.candi) + (uint32_t)warp * (M3_WCAP * 4u);
      const uint32_t kb1m = kh > 0 ? kb1 : 0x10000u, span1 = ke1 - kb1, h1a = smem_u32(&sm.hist[1][0]);   // kh == 0: no bracket
      // Warp w streams the contiguous slice [ws, we) of the row's vectors, 4 x 32 vectors (2 KB) per step, so that its
      // region of the candidate buffer is in ascending index order and regions follow each other in index order: the rank
      // of a value among equal values (index ascending) is a count over earlier regions plus a running count.
      // FULL: all four vectors of every lane lie inside the slice.
      const long long per = (nv + M3_WARPS - 1) / M3_WARPS, ws = warp * per < nv ? warp * per : nv, we = ws + per < nv ? ws + per : nv;
      auto chunk = [&](const long long v0, auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
        if (lane == 0) {   // the step three ahead goes to L2 now
          const long long pv = v0 + 3 * 128;
          if (pv < we) m3_prefetch_l2(src + pv, (uint32_t)((we - pv < 128 ? we - pv : 128) * 16));
        }
        uint4 q[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const long long v = v0 + u * 32 + lane;
          q[u] = make_uint4(0u, 0u, 0u, 0u);
          if (FULL || v < we) q[u] = __ldg(src + v);
        }
        // candidate masks of the four vectors: bit 2 j + half of mv[u] = value `half` of word j of vector u
        uint32_t mv[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const long long v = v0 + u * 32 + lane;
          const uint32_t w4[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
          uint32_t cm[4], gm[4];
#pragma unroll
          for (int e = 0; e < 4; e++) {
            const __half2 h = *reinterpret_cast<const __half2*>(&w4[e]);
            gm[e] = __hgt2_mask(h, hmhi);
            cm[e] = __hgeu2_mask(h, htop) | __hle2_mask(h, hbot) | (__hge2_mask(h, hmlo) & ~gm[e]);
          }
          mv[u] = 0;
          if (FULL || v < we) {   // lanes beyond the slice hold zeros and must stay out
            // count above the bracket: every true half of a compare mask is two 0xFF bytes, dp4a adds 2 x 255 (no alu op)
#pragma unroll
            for (int e = 0; e < 4; e++) gacc = __dp4a(gm[e], 0x01010101u, gacc);
            // the eight candidate flags as bits: byte 0 / 2 of each mask word are -1 or 0, dp4a weighs them 1, 2, 4, ...
            mv[u] = (uint32_t)(-m3_dp4a_su(__byte_perm(cm[0], cm[1], 0x6420u), 0x08040201u,
                                           m3_dp4a_su(__byte_perm(cm[2], cm[3], 0x6420u), 0x80402010u, 0)));
          }
        }
        // slots in index order: vector u of every lane before vector u + 1 of any lane; two packed scans per step
        const uint32_t c0 = __popc(mv[0]), c1 = __popc(mv[1]), c2 = __popc(mv[2]), c3 = __popc(mv[3]);
        const uint32_t i01 = m3_warp_inclusive(c0 | (c1 << 16), lane), i23 = m3_warp_inclusive(c2 | (c3 << 16), lane);
        const uint32_t t01 = __shfl_sync(0xffffffffu, i01, 31), t23 = __shfl_sync(0xffffffffu, i23, 31);
        uint32_t posv[4];
        posv[0] = wcnt + (i01 & 0xFFFFu) - c0;
        posv[1] = wcnt + (t01 & 0xFFFFu) + (i01 >> 16) - c1;
        posv[2] = wcnt + (t01 & 0xFFFFu) + (t01 >> 16) + (i23 & 0xFFFFu) - c2;
        posv[3] = wcnt + (t01 & 0xFFFFu) + (t01 >> 16) + (t23 & 0xFFFFu) + (i23 >> 16) - c3;
        wcnt += (t01 & 0xFFFFu) + (t01 >> 16) + (t23 & 0xFFFFu) + (t23 >> 16);
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const uint32_t w0 = q[u].x, w1 = q[u].y, w2 = q[u].z, w3 = q[u].w;
          const uint32_t vtag = (uint32_t)(v0 + u * 32 + lane) << 8;
          uint32_t m = mv[u];
          uint32_t pos = posv[u];
          while (m) {   // no index arithmetic on the way: the candidate is named by its one-hot bit
            const uint32_t b = m & (0u - m);
            m ^= b;
            const bool upper = (b & 0xF0u) != 0;
            const uint32_t a = upper ? w2 : w0, c = upper ? w3 : w1;
            const uint32_t w = (b & 0xCCu) ? c : a;
            const uint32_t val = (b & 0xAAu) ? (w >> 16) : (w & 0xFFFFu);
            const uint32_t d = mn_dkey(val);
            const uint32_t t = d - kb1m;
            // the key and (vector << 8 | bit) go to the warp's region (nothing is stored beyond its end: a warp that
            // overflows is caught below); a member of the median bracket is counted in its level-1 histogram right
            // here (the shared-memory atomics hide under the stream instead of piling up in step C)
            asm volatile(
                "{\n\t.reg .pred p, q;\n\tsetp.lt.u32 p, %7, %8;\n\tsetp.le.u32 q, %4, %5;\n\t"
                "@p st.shared.u16 [%0], %1;\n\t@p st.shared.u32 [%2], %3;\n\t@q red.shared.add.u32 [%6], 1;\n\t}" ::"r"(ka + pos * 2u),
                "h"((unsigned short)d), "r"(ia + pos * 4u), "r"(vtag | b), "r"(t), "r"(span1), "r"(h1a + ((t >> sh1) << 2)),
                "r"(pos), "r"((uint32_t)M3_WCAP)
                : "memory");
            pos++;
          }
        }
      };
      {
        long long v0 = ws;
        for (; v0 + 128 <= we; v0 += 128) chunk(v0, std::true_type{});
        if (v0 < we) chunk(v0, std::false_type{});
      }
      // the last n % 8 values: the end of the last warp's slice
      if (tid == (M3_WARPS - 1) * 32) {
        for (long long i = nv * 8; i < n; i++) {
          const unsigned short bits = src16[i];
          const __half h = __ushort_as_half(bits);
          if (__hgt(h, smhi)) gcount++;
          if (__hgeu(h, stop) || __hle(h, sbot) || (__hge(h, smlo) && !__hgt(h, smhi))) {
            const uint32_t pos = wcnt;
            const uint32_t d = mn_dkey(bits);
            if (pos < (uint32_t)M3_WCAP) {
              sm.candk[(M3_WARPS - 1) * M3_WCAP + pos] = (unsigned short)d;
              sm.candi[(M3_WARPS - 1) * M3_WCAP + pos] = ((uint32_t)(i >> 3) << 8) | (1u << (i & 7));
            }
            if (d - kb1m <= span1) atomicAdd(&sm.hist[1][(d - kb1m) >> sh1], 1u);
            wcnt++;
          }
        }
      }
      wcnt = __shfl_sync(0xffffffffu, wcnt, 0);
      gcount += gacc / 510u;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) gcount += __shfl_xor_sync(0xffffffffu, gcount, o);
      if (lane == 0) {
        atomicAdd(&sm.G, gcount);
        sm.wcount[warp] = wcnt;
      }
    }
    __syncthreads();

    // ---- C: exact selection among the candidates, the three classes side by side ----
    // class 0: values >= T_top, window = its first k;  class 1: the bracket of the median, window = ranks m0 - G ..
    // m1 - 1 - G;  class 2: values <= T_bot, window = its last k.  Per class a two-level radix select over the key
    // range [kbase, kend] (+0 / -0 compare equal: a range that ends at one of them is widened over both), then a rank
    // sort of the keys that remain.
    if (row + gridDim.x < p.rows) {   // the next row of this CTA: sample sectors and the first chunks on their way to L2
      const long long nrow = row + gridDim.x;
      const uint4* nsrc = reinterpret_cast<const uint4*>(p.vals + nrow * p.row_stride);
      if (lane == 0) {   // the first three steps of this warp's slice
        const long long per = (nv + M3_WARPS - 1) / M3_WARPS, ws = warp * per < nv ? warp * per : nv, we = ws + per < nv ? ws + per : nv;
        if (ws < we) m3_prefetch_l2(nsrc + ws, (uint32_t)((we - ws < 384 ? we - ws : 384) * 16));
      }
      for (long long g = tid; g < ngroups; g += M3_THREADS) {
        const long long sector = (g << slog) + (m3_hash((uint32_t)g, (uint32_t)nrow) >> (32 - slog));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(nsrc + sector * 2));
      }
    }
    const uint32_t G = sm.G;
    bool ok = true;
#pragma unroll
    for (int w = 0; w < M3_WARPS; w++) ok = ok && sm.wcount[w] <= (uint32_t)M3_WCAP;
    // this warp's candidates: slots wb .. wb + wn
    const uint32_t wb = (uint32_t)warp * M3_WCAP, wn = ok ? sm.wcount[warp] : 0u;
    // C1: level-1 histograms of the two tail classes (the buffer holds keys; NaN keys lie beyond the two infinities)
    const uint32_t wend = wb + wn;
    for (uint32_t i0 = wb + lane; i0 < wend; i0 += 128) {
      uint32_t d[4];
#pragma unroll
      for (int j = 0; j < 4; j++) d[j] = i0 + 32 * j < wend ? (uint32_t)sm.candk[i0 + 32 * j] : 0x8000u;   // -0: in no tail class
#pragma unroll
      for (int j = 0; j < 4; j++) {
        if (i0 + 32 * j < wend && (d[j] <= ke0 || d[j] >= kb2)) {   // one candidate in eight; NaN keys are tail keys
          if (d[j] < 0x3FFu || d[j] > 0xFC00u) sm.nan = 1u;
          if (d[j] <= ke0) atomicAdd(&sm.hist[0][(d[j] - kb0) >> sh0], 1u);
          if (d[j] >= kb2) atomicAdd(&sm.hist[2][(d[j] - kb2) >> sh2], 1u);
        }
      }
    }
    __syncthreads();
    ok = ok && sm.nan == 0;
    // C2: prefix sums, the bins of each window's first and last rank
    uint32_t rl0 = 0, rl1 = 0, rl2 = 0, rh0 = 0, rh1 = 0, rh2 = 0;
    {
      uint32_t cb[3][4], tot[3], inc[3];
#pragma unroll
      for (int c = 0; c < 3; c++) {
        tot[c] = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) { cb[c][i] = sm.hist[c][tid * 4 + i]; tot[c] += cb[c][i]; }
        inc[c] = m3_warp_inclusive(tot[c], lane);
        if (lane == 31) sm.scan[c][warp] = inc[c];
      }
      __syncthreads();
#pragma unroll
      for (int c = 0; c < 3; c++) {
        uint32_t ex = inc[c] - tot[c], total = 0;
#pragma unroll
        for (int w = 0; w < M3_WARPS; w++) {
          const uint32_t sw = sm.scan[c][w];
          ex += w < warp ? sw : 0u;
          total += sw;
        }
        uint32_t rl, rh;
        if (c == 1) {
          if (kh == 0) continue;
          if ((long long)G > m0 || (long long)G + (long long)total < m1) { ok = false; continue; }
          rl = (uint32_t)(m0 - (long long)G); rh = (uint32_t)(m1 - 1 - (long long)G);
          rl1 = rl; rh1 = rh;
        } else {
          if (total < (uint32_t)k) { ok = false; continue; }
          rl = c == 0 ? 0u : total - (uint32_t)k; rh = rl + (uint32_t)k - 1u;
          if (c == 0) { rl0 = rl; rh0 = rh; } else { rl2 = rl; rh2 = rh; }
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const uint32_t in = ex + cb[c][i];
          if (ex <= rl && rl < in) { sm.binA[c] = (uint32_t)tid * 4 + i; sm.exA[c] = ex; }
          if (ex <= rh && rh < in) { sm.binB[c] = (uint32_t)tid * 4 + i; sm.exB[c] = ex; }
          ex = in;
        }
      }
    }
    __syncthreads();
    if (ok) {   // block-uniform
      // C3: the low key bits inside the boundary bins (first key of bin A / B of each class)
      const uint32_t fa0 = kb0 + (sm.binA[0] << sh0), fb0 = kb0 + (sm.binB[0] << sh0);
      const uint32_t fa1 = kb1 + (sm.binA[1] << sh1), fb1 = kb1 + (sm.binB[1] << sh1);
      const uint32_t fa2 = kb2 + (sm.binA[2] << sh2), fb2 = kb2 + (sm.binB[2] << sh2);
      if (sh0 | sh1 | sh2) {
        const uint32_t w0 = 1u << sh0, w1 = 1u << sh1, w2 = 1u << sh2;
        const bool l1 = sh1 > 0 && kh > 0, l0 = sh0 > 0, l2 = sh2 > 0;
        for (uint32_t i0 = wb + lane; i0 < wend; i0 += 128) {
          uint32_t d[4];
#pragma unroll
          for (int j = 0; j < 4; j++) d[j] = i0 + 32 * j < wend ? (uint32_t)sm.candk[i0 + 32 * j] : 0xFFFFFFFFu;
#pragma unroll
          for (int j = 0; j < 4; j++) {
            if (i0 + 32 * j >= wend) continue;
            if (l1) {
              if (d[j] - fa1 < w1) atomicAdd(&sm.h2[1][0][d[j] - fa1], 1u);
              if (d[j] - fb1 < w1) atomicAdd(&sm.h2[1][1][d[j] - fb1], 1u);
            }
            if (l0) {
              if (d[j] - fa0 < w0) atomicAdd(&sm.h2[0][0][d[j] - fa0], 1u);
              if (d[j] - fb0 < w0) atomicAdd(&sm.h2[0][1][d[j] - fb0], 1u);
            }
            if (l2) {
              if (d[j] - fa2 < w2) atomicAdd(&sm.h2[2][0][d[j] - fa2], 1u);
              if (d[j] - fb2 < w2) atomicAdd(&sm.h2[2][1][d[j] - fb2], 1u);
            }
          }
        }
        __syncthreads();
      }
      // C4: warp 2 c + b resolves boundary b of class c
      if (warp < 6) {
        const int c = warp >> 1, b = warp & 1;
        const int sh = (int)m3_sel3(c, sh0, sh1, sh2);
        const uint32_t exb = b ? sm.exB[c] : sm.exA[c];
        const uint32_t r = b ? m3_sel3(c, rh0, rh1, rh2) : m3_sel3(c, rl0, rl1, rl2);
        uint32_t key = b ? m3_sel3(c, fb0, fb1, fb2) : m3_sel3(c, fa0, fa1, fa2), less = exb;
        if (sh > 0) {
          const uint32_t cnt = lane < (1 << sh) ? sm.h2[c][b][lane] : 0u;
          const uint32_t inc = m3_warp_inclusive(cnt, lane);
          const bool mine = exb + inc - cnt <= r && r < exb + inc;
          const uint32_t sel = __ballot_sync(0xffffffffu, mine);
          const int j = sel ? __ffs(sel) - 1 : 0;
          key += (uint32_t)j;
          less = exb + __shfl_sync(0xffffffffu, inc - cnt, j);
        }
        if (lane == 0) {
          if (b == 0) { sm.klo[c] = key; sm.less_lo[c] = less; } else { sm.khi[c] = key; sm.less_hi[c] = less; }
        }
      }
      __syncthreads();
      // C5: the members of the three windows.  A key strictly between the boundary keys is in; a key EQUAL to a boundary
      // key is in according to its rank among the equal values in index order: regions are in index order (step B), so
      // that rank is (equal values in earlier warps' regions) + (equal values earlier in this region).
      const uint32_t kl0 = sm.klo[0], kl1 = sm.klo[1], kl2 = sm.klo[2];
      const uint32_t kh0 = sm.khi[0], kh1 = sm.khi[1], kh2 = sm.khi[2];
      const uint32_t sp0 = kh0 - kl0, sp1 = kh > 0 ? kh1 - kl1 : 0u, sp2 = kh2 - kl2;
      const uint32_t K[6] = {kl0, kh0, kl1, kh1, kl2, kh2};
      // First the few per cent of the region whose keys lie inside a window's key range are compacted, in order, into a
      // short list per warp (the level-1 histograms are free by now and hold the lists): the tie counts and the member
      // pass then run over ~20-150 entries per warp instead of ~470.
      constexpr uint32_t SL = 256;                                   // short-list entries per warp: key << 16 | position in the region
      uint32_t* const sl = &sm.hist[0][0] + (uint32_t)warp * SL;     // 16 x 256 words = hist[0] and hist[1]
      const uint32_t ltm = (1u << lane) - 1u;
      uint32_t nsl = 0;                                              // warp-uniform
      for (uint32_t i0 = wb + lane; i0 - lane < wend; i0 += 128) {   // warp-uniform trip count, region order
        uint32_t d[4];
#pragma unroll
        for (int j = 0; j < 4; j++) d[j] = i0 + 32 * j < wend ? (uint32_t)sm.candk[i0 + 32 * j] : 0xFFFFFFFFu;
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const bool inr = i0 + 32 * j < wend && (d[j] - kl0 <= sp0 || (kh > 0 && d[j] - kl1 <= sp1) || d[j] - kl2 <= sp2);
          const uint32_t bal = __ballot_sync(0xffffffffu, inr);
          if (bal == 0) continue;
          const uint32_t slot = nsl + __popc(bal & ltm);
          if (inr && slot < SL) sl[slot] = (d[j] << 16) | (i0 + 32 * j - wb);
          nsl += __popc(bal);
        }
      }
      __syncwarp();
      const uint32_t nslc = nsl < SL ? nsl : SL;
      {   // per-warp counts of the six boundary keys
        uint32_t cn[6] = {0, 0, 0, 0, 0, 0};
        for (uint32_t t = lane; t < nslc; t += 32) {
          const uint32_t d = sl[t] >> 16;
#pragma unroll
          for (int q = 0; q < 6; q++) cn[q] += d == K[q];
        }
#pragma unroll
        for (int h = 0; h < 3; h++) {   // two counts per word (a count is < 2^14)
          uint32_t pk = cn[2 * h] | (cn[2 * h + 1] << 16);
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) pk += __shfl_xor_sync(0xffffffffu, pk, o);
          if (lane == 0) { sm.tie[2 * h][warp] = pk & 0xFFFFu; sm.tie[2 * h + 1][warp] = pk >> 16; }
        }
        if (lane == 0 && nsl > SL) sm.nan = 2u;   // the short list overflowed (a tie group of thousands): the row falls back
      }
      __syncthreads();
      if (sm.nan != 0) ok = false;
      uint32_t run[6];                                  // equal values before the current position (warp-uniform)
      {   // lane w holds the counts of warp w, two keys per word; the warps before this one are summed
        uint32_t pk[3];
#pragma unroll
        for (int h = 0; h < 3; h++) {
          pk[h] = lane < warp ? (sm.tie[2 * h][lane & (M3_WARPS - 1)] | (sm.tie[2 * h + 1][lane & (M3_WARPS - 1)] << 16)) : 0u;
#pragma unroll
          for (int o = 8; o > 0; o >>= 1) pk[h] += __shfl_xor_sync(0xffffffffu, pk[h], o);
          pk[h] = __shfl_sync(0xffffffffu, pk[h], 0);
          run[2 * h] = pk[h] & 0xFFFFu; run[2 * h + 1] = pk[h] >> 16;
        }
      }
      // tie ranks [lo_from, lo_to) of klo and [0, hi_to) of khi belong to the window (klo == khi: one group holds both ends)
      const uint32_t s0 = rl0 - sm.less_lo[0], s1 = rl1 - sm.less_lo[1], s2 = rl2 - sm.less_lo[2];
      const uint32_t lo_from[3] = {s0, s1, s2};
      const uint32_t lo_to[3] = {kl0 == kh0 ? s0 + (rh0 - rl0 + 1u) : 0xFFFFFFFFu, kl1 == kh1 ? s1 + (rh1 - rl1 + 1u) : 0xFFFFFFFFu,
                                 kl2 == kh2 ? s2 + (rh2 - rl2 + 1u) : 0xFFFFFFFFu};
      const uint32_t hi_to[3] = {rh0 - sm.less_hi[0] + 1u, rh1 - sm.less_hi[1] + 1u, rh2 - sm.less_hi[2] + 1u};
      for (uint32_t t0 = 0; ok && t0 < nslc; t0 += 32) {   // warp-uniform trip count, region order
        const bool live = t0 + lane < nslc;
        const uint32_t ent = live ? sl[t0 + lane] : 0xFFFFFFFFu;
        const uint32_t d = live ? ent >> 16 : 0xFFFFFFFFu;
        bool in[3] = {live && d - kl0 <= sp0, live && kh > 0 && d - kl1 <= sp1, live && d - kl2 <= sp2};
        const bool eq = d == K[0] || d == K[1] || d == K[2] || d == K[3] || d == K[4] || d == K[5];
        if (__any_sync(0xffffffffu, eq)) {
#pragma unroll
          for (int c = 0; c < 3; c++) {
            const bool elo = in[c] && d == K[2 * c], ehi = in[c] && d == K[2 * c + 1] && K[2 * c] != K[2 * c + 1];
            const uint32_t blo = __ballot_sync(0xffffffffu, elo), bhi = __ballot_sync(0xffffffffu, ehi);
            if (elo) { const uint32_t t = run[2 * c] + __popc(blo & ltm); in[c] = t >= lo_from[c] && t < lo_to[c]; }
            if (ehi) { const uint32_t t = run[2 * c + 1] + __popc(bhi & ltm); in[c] = t < hi_to[c]; }
            run[2 * c] += __popc(blo); run[2 * c + 1] += __popc(bhi);
          }
        }
        if (!(in[0] | in[1] | in[2])) continue;
        const uint32_t cw = sm.candi[wb + (ent & 0xFFFFu)];
        const uint32_t ci = (cw >> 8) * 8u + (uint32_t)(__ffs(cw & 0xFFu) - 1);   // vector << 8 | one-hot bit -> index
        if (in[1]) {
          const uint32_t slt = atomicAdd(&sm.lcount[1], 1u);
          if (slt < (uint32_t)M3_LIST) sm.lk[1][slt] = ((unsigned long long)d << 32) | ci;
        }
        if (in[0]) {
          const uint32_t slt = atomicAdd(&sm.lcount[0], 1u);
          if (slt < (uint32_t)M3_LIST) sm.lk[0][slt] = ((unsigned long long)d << 32) | ci;
        }
        if (in[2]) {
          const uint32_t slt = atomicAdd(&sm.lcount[2], 1u);
          if (slt < (uint32_t)M3_LIST) sm.lk[2][slt] = ((unsigned long long)d << 32) | ci;
        }
      }
      __syncthreads();
      if (sm.lcount[0] > (uint32_t)M3_LIST || sm.lcount[2] > (uint32_t)M3_LIST || (kh > 0 && sm.lcount[1] > (uint32_t)M3_LIST)) {
        ok = false;   // cannot happen: a list holds exactly its window
      }
      if (ok) {
        // C6: rank sorts, five warps per class: packed (key, index) ascending = value descending, index ascending
        const int c = tid / M3_SORT_THREADS;
        if (c < 3 && (c != 1 || kh > 0)) {
          const int cnt = (int)sm.lcount[c];
          const uint32_t rl = m3_sel3(c, rl0, rl1, rl2), rh = m3_sel3(c, rh0, rh1, rh2);
          const int size = (int)(rh - rl + 1u);   // the list holds exactly the window (step C5)
          int* io = p.idx_out + (row * 3 + c) * (long long)k;
          __half* vo = p.val_out ? p.val_out + (row * 3 + c) * (long long)k : nullptr;
          const unsigned long long* list = sm.lk[c];
          for (int t = tid - c * M3_SORT_THREADS; t < cnt; t += M3_SORT_THREADS) {
            const unsigned long long mine = list[t];
            int r = 0;
            int o = 0;
#pragma unroll 4
            for (; o + 2 <= cnt; o += 2) {
              const ulonglong2 ot = *reinterpret_cast<const ulonglong2*>(list + o);
              r += (ot.x < mine) + (ot.y < mine);
            }
            for (; o < cnt; o++) r += list[o] < mine;
            if (r < size) {
              io[r] = (int)(uint32_t)mine;
              if (vo) vo[r] = __ushort_as_half((unsigned short)mn_bits((uint32_t)(mine >> 32)));
            }
          }
          for (int t = size + tid - c * M3_SORT_THREADS; t < k; t += M3_SORT_THREADS) {
            io[t] = -1;
            if (vo) vo[t] = __ushort_as_half((unsigned short)0);
          }
        }
        if (kh == 0 && tid < k) {
          p.idx_out[(row * 3 + 1) * (long long)k + tid] = -1;
          if (p.val_out) p.val_out[(row * 3 + 1) * (long long)k + tid] = __ushort_as_half((unsigned short)0);
        }
      }
    }
    if (!ok && tid == 0) {
      const int slot = atomicAdd(p.fb_count, 1);
      p.fb_list[slot] = (int)row;
    }
    __syncthreads();
  }
}

}  // namespace rq
