// C ABI of librqae_b200.so (declared in include/rqae_b200.h): weight packing, kernel selection and
// launch.  Host logic only; the kernels live in rq_forward.cuh / rq_decode.cuh.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <condition_variable>
#include <map>
#include <mutex>
#include <thread>
#include <tuple>
#include <vector>
#include <math.h>
#if defined(__x86_64__) && !defined(RQ_NO_STREAM)
#include <immintrin.h>
#endif

#include "../../include/rqae_b200.h"
#include "rq_decode.cuh"
#include "rq_forward.cuh"
#include "rq_intensity.cuh"
#include "rq_intensity_exact.cuh"
#include "rq_mine.cuh"
#include "rq_mine3.cuh"
#include "rq_search.cuh"
#include "rq_layout.h"

#ifndef RQ_L2_HOT_DEFAULT
#define RQ_L2_HOT_DEFAULT 1.0f
#endif

namespace {

// Lock-step counters of the forward kernel (rq_forward.cuh, "grid lock-step"): one slot per launch in flight.
constexpr int kSyncSlots = 64;
__device__ unsigned int g_sync_ctr[kSyncSlots * 32];   // 128 bytes apart
std::atomic<unsigned int> g_launch_seq{0};
std::atomic<int> g_forward_variant{-1};   // -1: not initialised (RQAE_CLUSTER), 0: single-CTA units, 1: D-split clusters where built

thread_local cudaError_t g_last_cuda = cudaSuccess;
thread_local int64_t g_launches = 0;

#define RQ_CUDA(call)                    \
  do {                                   \
    cudaError_t e__ = (call);            \
    if (e__ != cudaSuccess) {            \
      g_last_cuda = e__;                 \
      return RQAE_ECUDA;                 \
    }                                    \
  } while (0)

// Counts a kernel launch that the runtime accepted (rqae_launch_count) and returns the launch's error.
cudaError_t launched(cudaError_t e = cudaGetLastError()) {
  if (e == cudaSuccess) g_launches++;
  return e;
}

// Set a function attribute of a kernel once per (kernel, attribute, device) and remember the result: attributes are
// per device, and a process may drive more than one.
cudaError_t ensure_func_attr(const void* kern, cudaFuncAttribute attr, int value) {
  static std::mutex mu;
  static std::map<std::tuple<const void*, int, int>, cudaError_t> done;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(mu);
  const auto key = std::make_tuple(kern, (int)attr, dev);
  auto it = done.find(key);
  if (it != done.end()) return it->second;
  return done[key] = cudaFuncSetAttribute(kern, attr, value);
}

// Calls f with a value of the C++ type of code_dtype (RQAE_CODE_*): the kernels that read codes are templates on it.
template <typename F>
void with_code_type(int code_dtype, F&& f) {
  if (code_dtype == RQAE_CODE_I64) f((long long)0);
  else if (code_dtype == RQAE_CODE_I32) f((int)0);
  else f((short)0);
}

// A stream-ordered pool of this library's own per device, for the few bytes per row of the selection's fallback list.
// The default pool gives unused memory back at every synchronisation (release threshold 0), so the first call after
// a sync would pay an allocation from the driver; this pool keeps what it has.
cudaError_t scratch_pool(cudaMemPool_t* out) {
  static std::mutex mu;
  static std::map<int, cudaMemPool_t> pools;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(mu);
  auto it = pools.find(dev);
  if (it == pools.end()) {
    cudaMemPoolProps props = {};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    cudaMemPool_t pool;
    e = cudaMemPoolCreate(&pool, &props);
    if (e != cudaSuccess) return e;
    unsigned long long keep = ~0ull;
    e = cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    if (e != cudaSuccess) return e;
    it = pools.emplace(dev, pool).first;
  }
  *out = it->second;
  return cudaSuccess;
}

int device_sm_count(int* sms) {
  int dev = 0;
  RQ_CUDA(cudaGetDevice(&dev));
  int major = 0;
  RQ_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) return RQAE_ENODEVICE;
  RQ_CUDA(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
  return RQAE_OK;
}

// ---------------------------------------------------------------------------------------------
// packing kernels
// ---------------------------------------------------------------------------------------------
__global__ void pack_stages_kernel(const float* __restrict__ w_in, const float* __restrict__ b_in,
                                   const float* __restrict__ w_out, const float* __restrict__ b_out, int nq, int D,
                                   int E, int CH, unsigned char* __restrict__ packed, size_t off_bin,
                                   size_t off_stage, size_t stage_bytes) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_stage = (long long)E * RQ_GROUP_THREADS;
  const long long total = (long long)(nq + 1) * per_stage;
  if (gid < nq + 1) {
    float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
    if (gid < nq) b = make_float4(b_in[gid * 4 + 0], b_in[gid * 4 + 1], b_in[gid * 4 + 2], b_in[gid * 4 + 3]);
    reinterpret_cast<float4*>(packed + off_bin)[gid] = b;
  }
  if (gid >= total) return;
  const int s = (int)(gid / per_stage);
  const int rem = (int)(gid % per_stage);
  const int j = rem / RQ_GROUP_THREADS, t = rem % RQ_GROUP_THREADS;
  const int JC = E / CH;
  const int c = j / JC, jj = j % JC;
  const int d = j * RQ_GROUP_THREADS + t;
  unsigned char* chunk = packed + off_stage + (size_t)s * stage_bytes + (size_t)c * (stage_bytes / CH);
  float4 wo = make_float4(0.f, 0.f, 0.f, 0.f), wi = wo;
  float bo = 0.f;
  if (d < D) {
    if (s >= 1) {
      const float* w = w_out + ((size_t)(s - 1) * D + d) * 4;
      wo = make_float4(w[0], w[1], w[2], w[3]);
      bo = b_out[(size_t)(s - 1) * D + d];
    }
    if (s < nq) {
      const float* w = w_in + (size_t)s * 4 * D + d;
      // component c holds k = c ^ (t & 3): see butterfly32 in rq_forward.cuh
      const int x = t & 3;
      wi = make_float4(w[(size_t)(0 ^ x) * D], w[(size_t)(1 ^ x) * D], w[(size_t)(2 ^ x) * D], w[(size_t)(3 ^ x) * D]);
    }
  }
  const size_t e = (size_t)jj * RQ_GROUP_THREADS + t;
  reinterpret_cast<float4*>(chunk)[e] = wo;
  reinterpret_cast<float4*>(chunk + (size_t)JC * RQ_GROUP_THREADS * 16)[e] = wi;
  reinterpret_cast<float*>(chunk + (size_t)JC * RQ_GROUP_THREADS * 32)[e] = bo;
}

// Search tables for the shared-codebook mode, built on the host (the table is a few KB; this runs once per
// weight load).
//  (1) De-duplicated table: rows that are value-identical to an earlier row are dropped (torch.argmax
//      returns the first maximum, so a later duplicate can never be selected); the original index of every
//      surviving row is kept; padded to a multiple of 32 with copies of row 0 (a copy ties with row 0 and
//      loses on the position).
//  (2) Canonical-row tables, built when the table is closed under flipping the sign of any coordinate and
//      under exchanging any two coordinates (true for the fsq / round_fsq grids).  Then for a query z
//          max_k z.c_k  is attained by a row whose signs follow z and whose magnitudes are ordered like |z|
//      (rearrangement inequality), i.e. by a *canonical* row c0 >= c1 >= c2 >= c3 >= 0 re-arranged to the
//      magnitude order of z: 10 candidates instead of 625 for round_fsq 5^4.  tp[order][r] holds canonical
//      row r with its coordinates placed per `order` (the Lehmer code of the magnitude ranks, see
//      rq_forward.cuh); map3[signs][order][r] is the lowest original index of the resulting signed row.
//      The thresholds bound when this shortcut provably returns the reference's first maximum (DESIGN.md,
//      "Search"); any token outside them takes the exhaustive scan in the reference's own arithmetic.
struct SearchTables {
  RqHeader hdr;
  std::vector<float> cbt;
  std::vector<unsigned short> map;
  std::vector<float> tp;
  std::vector<unsigned short> map3;
};

typedef std::array<uint32_t, 4> RowKey;
static RowKey row_key(const float* v) {
  RowKey k;
  for (int i = 0; i < 4; i++) {
    float f = v[i] == 0.f ? 0.f : v[i];   // -0 -> +0
    memcpy(&k[i], &f, 4);
  }
  return k;
}

static int lehmer_order(const float* a) {   // a = magnitudes; must match the kernel's formula
  const int c01 = a[1] > a[0], c02 = a[2] > a[0], c03 = a[3] > a[0], c12 = a[2] > a[1], c13 = a[3] > a[1], c23 = a[3] > a[2];
  return 6 * (c01 + c02 + c03) + 2 * (c12 + c13) + c23;
}

static void build_search_tables(const float* cb, int K, int KT, SearchTables* T) {
  memset(&T->hdr, 0, sizeof(T->hdr));
  T->cbt.assign((size_t)KT * 4, 0.f);
  T->map.assign((size_t)KT, 0);
  T->tp.assign((size_t)RQ_NPERM * RQ_CAN_MAX * 4, 0.f);
  T->map3.assign((size_t)RQ_NSIGN * RQ_NPERM * RQ_CAN_MAX, 0);
  std::map<RowKey, int> first;   // value -> lowest original index
  std::vector<int> keep;
  bool finite = true;
  float cmin = INFINITY, n2max = 0.f;
  for (int k = 0; k < K; k++) {
    const float* r = cb + (size_t)k * 4;
    float n2 = 0.f;
    for (int i = 0; i < 4; i++) {
      const float m = fabsf(r[i]);
      if (!(m <= 3.0e38f)) finite = false;
      if (m > 0.f && m < cmin) cmin = m;
      n2 += m * m;
    }
    if (n2 > n2max) n2max = n2;
    if (first.emplace(row_key(r), k).second) keep.push_back(k);
  }
  int n = 0;
  for (int k : keep) { memcpy(&T->cbt[(size_t)n * 4], cb + (size_t)k * 4, 16); T->map[n] = (unsigned short)k; n++; }
  const int kd = n, kd_pad = (kd + 31) / 32 * 32;
  for (; n < kd_pad && n < KT; n++) { memcpy(&T->cbt[(size_t)n * 4], &T->cbt[0], 16); T->map[n] = T->map[0]; }
  T->hdr.kd = kd;
  T->hdr.kd_pad = kd_pad;
  if (!finite || !(cmin < INFINITY) || K > 16384) return;
  // closure under the generators of the hyperoctahedral group: 4 sign flips, 3 adjacent transpositions
  for (int k : keep) {
    const float* r = cb + (size_t)k * 4;
    for (int i = 0; i < 4; i++) {
      float f[4] = {r[0], r[1], r[2], r[3]};
      f[i] = -f[i];
      if (!first.count(row_key(f))) return;
    }
    for (int i = 0; i < 3; i++) {
      float f[4] = {r[0], r[1], r[2], r[3]};
      const float t = f[i]; f[i] = f[i + 1]; f[i + 1] = t;
      if (!first.count(row_key(f))) return;
    }
  }
  // canonical rows (ascending original index), zero row excluded
  std::vector<int> can;
  float dmin = INFINITY;
  for (int k : keep) {
    const float* r = cb + (size_t)k * 4;
    if (r[0] >= r[1] && r[1] >= r[2] && r[2] >= r[3] && r[3] >= 0.f && r[0] > 0.f) {
      can.push_back(k);
      const float seq[5] = {r[0], r[1], r[2], r[3], 0.f};
      for (int i = 0; i < 4; i++)
        if (seq[i] != seq[i + 1] && seq[i] - seq[i + 1] < dmin) dmin = seq[i] - seq[i + 1];
    }
  }
  if (can.empty() || (int)can.size() > RQ_CAN_MAX || !(dmin < INFINITY)) return;
  int rank[4] = {0, 1, 2, 3};
  do {   // rank[i] = position of coordinate i in the descending magnitude order
    float a[4];
    for (int i = 0; i < 4; i++) a[i] = (float)(4 - rank[i]);
    const int ord = lehmer_order(a);
    for (size_t r = 0; r < can.size(); r++) {
      const float* m = cb + (size_t)can[r] * 4;
      float* dst = &T->tp[((size_t)ord * RQ_CAN_MAX + r) * 4];
      for (int i = 0; i < 4; i++) dst[i] = m[rank[i]];
      for (int sg = 0; sg < RQ_NSIGN; sg++) {
        float f[4];
        for (int i = 0; i < 4; i++) f[i] = ((sg >> i) & 1) ? -dst[i] : dst[i];
        auto itf = first.find(row_key(f));
        if (itf == first.end()) return;   // cannot happen for a closed table
        T->map3[((size_t)sg * RQ_NPERM + ord) * RQ_CAN_MAX + r] = (unsigned short)itf->second;
      }
    }
  } while (std::next_permutation(rank, rank + 4));
  const float nmax = fmaxf(sqrtf(n2max), 1.0f);
  // error budget, in units of |z| (DESIGN.md): the reference's sqrt + divide + 4-term fma chain moves a
  // score by <= 4.8e-7*nmax, our un-normalised fp32 score by <= 2.4e-7*nmax
  T->hdr.can_rows = ((int)can.size() + 3) / 4 * 4;
  T->hdr.thr_tiny = 1.0e-6f * nmax / cmin;   // sign-flipped twin loses by >= 2*tiny*cmin      (2x margin)
  T->hdr.thr_gap = 3.0e-6f * nmax;           // runner-up cannot overtake                        (2x margin)
  T->hdr.thr_sep = 2.5e-6f * nmax / dmin;    // coordinate-swapped twin loses by >= sep*dmin     (2.6x margin)
}

// ---------------------------------------------------------------------------------------------
// FP32-pipe probes (roofline denominators measured by bench.py)
// ---------------------------------------------------------------------------------------------
template <bool PACKED>
__global__ void __launch_bounds__(512, 1) fp32_probe_kernel(int iters, float* sink) {
  using namespace rq;
  const float s = 1.0f + 1e-7f * (float)(threadIdx.x & 7), t = 1e-9f * (float)threadIdx.x;
  if (PACKED) {
    u64 a[12];
#pragma unroll
    for (int i = 0; i < 12; i++) a[i] = pack2((float)i, (float)(i + 1));
    const u64 ss = pack2(s, s), tt = pack2(t, t);
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int u = 0; u < 8; u++)
#pragma unroll
        for (int i = 0; i < 12; i++) a[i] = fma2(a[i], ss, tt);
    }
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 12; i++) { float lo, hi; unpack2(a[i], lo, hi); acc += lo + hi; }
    if (acc == 12345.678f) sink[0] = acc;
  } else {
    float a[24];
#pragma unroll
    for (int i = 0; i < 24; i++) a[i] = (float)i;
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int u = 0; u < 8; u++)
#pragma unroll
        for (int i = 0; i < 24; i++) a[i] = __fmaf_rn(a[i], s, t);
    }
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 24; i++) acc += a[i];
    if (acc == 12345.678f) sink[0] = acc;
  }
}

// Probe modes 2 / 3: the operand patterns of the forward kernel's two sweeps with everything in registers
// (no shared-memory traffic, no barriers), 2 warps per scheduler as in the kernel: what the FMA pipe delivers
// for (scalar weight) x (token pair) + (pair) chains -- the register-operand ceiling of the kernel's inner loops.
__device__ __forceinline__ rq::u64 fma2v(rq::u64 a, rq::u64 b, rq::u64 c) {   // volatile: not hoisted out of the probe loop
  rq::u64 d;
  asm volatile("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
template <int MODE>
__global__ void __launch_bounds__(256, 1) fma_pattern_probe_kernel(int iters, float* sink, const float* src) {
  using namespace rq;
  u64 r[4][3], acc[4][4], cp[4][4];
  float w[12], b[3];
  int n = threadIdx.x;   // every register gets its own source element so that nothing is merged
#pragma unroll
  for (int i = 0; i < 12; i++) w[i] = src[n++ & 127];
#pragma unroll
  for (int i = 0; i < 3; i++) b[i] = src[n++ & 127];
#pragma unroll
  for (int pi = 0; pi < 4; pi++) {
#pragma unroll
    for (int e = 0; e < 3; e++) { r[pi][e] = pack2(src[n & 127], src[(n + 1) & 127]); n += 2; }
#pragma unroll
    for (int k = 0; k < 4; k++) { acc[pi][k] = pack2(src[n & 127], src[(n + 1) & 127]); n += 2; cp[pi][k] = pack2(src[n & 127], src[(n + 1) & 127]); n += 2; }
  }
  const u64 neg1 = pack2(-1.0f, -1.0f);
  for (int it = 0; it < iters; it++) {
    if (MODE == 2) {   // sweep 2: acc[pi][k] += w[e][k] * r[pi][e]
#pragma unroll
      for (int e = 0; e < 3; e++)
#pragma unroll
        for (int pi = 0; pi < 4; pi++)
#pragma unroll
          for (int k = 0; k < 4; k++) acc[pi][k] = fma2(pack2(w[e * 4 + k], w[e * 4 + k]), r[pi][e], acc[pi][k]);
    } else {           // sweep 1: o = fma chain over k; r -= o
#pragma unroll
      for (int e = 0; e < 3; e++)
#pragma unroll
        for (int pi = 0; pi < 4; pi++) {
          // first multiplicand is loop-carried (another residual pair) so that ptxas cannot hoist the chain
          u64 o = fma2v(pack2(w[e * 4], w[e * 4]), r[pi][(e + 1) % 3], pack2(b[e], b[e]));
          o = fma2v(pack2(w[e * 4 + 1], w[e * 4 + 1]), cp[pi][1], o);
          o = fma2v(pack2(w[e * 4 + 2], w[e * 4 + 2]), cp[pi][2], o);
          o = fma2v(pack2(w[e * 4 + 3], w[e * 4 + 3]), cp[pi][3], o);
          r[pi][e] = fma2v(o, neg1, r[pi][e]);
        }
    }
  }
  float a = 0.f;
#pragma unroll
  for (int pi = 0; pi < 4; pi++) {
#pragma unroll
    for (int k = 0; k < 4; k++) { float lo, hi; unpack2(acc[pi][k], lo, hi); a += lo + hi; }
#pragma unroll
    for (int e = 0; e < 3; e++) { float lo, hi; unpack2(r[pi][e], lo, hi); a += lo + hi; }
  }
  if (a == 12345.678f) sink[0] = a;
}

// ---------------------------------------------------------------------------------------------
// forward launch
// ---------------------------------------------------------------------------------------------
// Takes the next of the forward kernel's lock-step counters (one per launch in flight) and zeroes it on `st`.
cudaError_t lockstep_slot(cudaStream_t st, unsigned int** slot) {
  unsigned int* base = nullptr;
  cudaError_t e = cudaGetSymbolAddress((void**)&base, g_sync_ctr);
  if (e != cudaSuccess) return e;
  *slot = base + (g_launch_seq.fetch_add(1) % kSyncSlots) * 32;
  return cudaMemsetAsync(*slot, 0, sizeof(unsigned int), st);
}

template <int E, int EC, int CH, int NSLOT, int TG, bool DBG, bool HOOK = false>
int launch_forward_t(const rq::FwdParams& prm, int sms, cudaStream_t st) {
  using C = rq::FwdCfg<E, EC, CH, NSLOT, TG>;
  auto kern = rq::rq_forward_kernel<E, EC, CH, NSLOT, TG, DBG, HOOK>;
  RQ_CUDA(ensure_func_attr((const void*)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SM_TOTAL));
  const long long n_units = (prm.n_tokens + 2 * TG - 1) / (2 * TG);
  const int grid = (int)(n_units < sms ? n_units : sms);
  rq::FwdParams p2 = prm;
  p2.sync_ctr = nullptr;
  if (n_units > grid) {
    // more than one unit per CTA: keep the CTAs' weight streams in step.
    // The kernel spins on the counter, so all CTAs must be co-resident: cooperative launch guarantees it.
    RQ_CUDA(lockstep_slot(st, &p2.sync_ctr));
    void* args[] = {(void*)&p2};
    RQ_CUDA(launched(cudaLaunchCooperativeKernel((const void*)kern, dim3(grid), dim3(rq::kThreads), args, C::SM_TOTAL, st)));
  } else {
    kern<<<grid, rq::kThreads, C::SM_TOTAL, st>>>(p2);
    RQ_CUDA(launched());
  }
  return RQAE_OK;
}

// D-split cluster variant: CS CTAs per unit, launched as clusters (co-scheduled on one GPC) and cooperatively (the
// grid lock-step spins on a global counter, so every cluster must be resident).
template <int E, int EC, int CH, int NSLOT, int TG, bool DBG, int CS>
int launch_forward_cluster_t(const rq::FwdParams& prm, int sms, cudaStream_t st) {
  using C = rq::FwdCfg<E, EC, CH, NSLOT, TG, CS>;
  auto kern = rq::rq_forward_kernel<E, EC, CH, NSLOT, TG, DBG, false, CS>;
  RQ_CUDA(ensure_func_attr((const void*)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SM_TOTAL));
  static std::mutex mu;
  static std::map<int, int> max_clusters;   // per device
  int dev = 0;
  RQ_CUDA(cudaGetDevice(&dev));
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.blockDim = dim3(rq::kThreads);
  cfg.dynamicSmemBytes = C::SM_TOTAL;
  cfg.stream = st;
  cudaLaunchAttribute attrs[2];
  attrs[0].id = cudaLaunchAttributeClusterDimension;
  attrs[0].val.clusterDim.x = CS; attrs[0].val.clusterDim.y = 1; attrs[0].val.clusterDim.z = 1;
  attrs[1].id = cudaLaunchAttributeCooperative;
  attrs[1].val.cooperative = 1;
  cfg.attrs = attrs;
  int ncl = 0;
  {
    std::lock_guard<std::mutex> lock(mu);
    auto it = max_clusters.find(dev);
    if (it == max_clusters.end()) {
      cfg.gridDim = dim3((unsigned)(sms / CS * CS));
      cfg.numAttrs = 1;
      int n = 0;
      RQ_CUDA(cudaOccupancyMaxActiveClusters(&n, (const void*)kern, &cfg));
      if (n <= 0) return RQAE_EUNSUPPORTED;
      it = max_clusters.emplace(dev, n).first;
    }
    ncl = it->second;
  }
  const long long n_units = (prm.n_tokens + 2 * TG - 1) / (2 * TG);
  const int clusters = (int)(n_units < ncl ? n_units : ncl);
  rq::FwdParams p2 = prm;
  p2.sync_ctr = nullptr;
  const bool coop = n_units > clusters;
  if (coop) RQ_CUDA(lockstep_slot(st, &p2.sync_ctr));
  cfg.gridDim = dim3((unsigned)(clusters * CS));
  cfg.numAttrs = coop ? 2 : 1;
  RQ_CUDA(launched(cudaLaunchKernelEx(&cfg, kern, p2)));
  return RQAE_OK;
}

template <int E, int EC, int CH, int NSLOT, int TG, int CS>
int launch_forward_cluster(const rq::FwdParams& prm, int sms, cudaStream_t st) {
  if (prm.teacher != nullptr || prm.z_out != nullptr) return launch_forward_cluster_t<E, EC, CH, NSLOT, TG, true, CS>(prm, sms, st);
  return launch_forward_cluster_t<E, EC, CH, NSLOT, TG, false, CS>(prm, sms, st);
}

template <int E, int EC, int CH, int NSLOT, int TG>
int launch_forward(const rq::FwdParams& prm, int sms, cudaStream_t st) {
  if (prm.hs != nullptr) return launch_forward_t<E, EC, CH, NSLOT, TG, false, true>(prm, sms, st);
  if (prm.teacher != nullptr || prm.z_out != nullptr) return launch_forward_t<E, EC, CH, NSLOT, TG, true>(prm, sms, st);
  return launch_forward_t<E, EC, CH, NSLOT, TG, false>(prm, sms, st);
}

// ---------------------------------------------------------------------------------------------
// tcgen05 GEMM of the intensities, the tensor-core decode and the tensor-core search maxima (rq_intensity.cuh)
// ---------------------------------------------------------------------------------------------
// Workspace of the intensity and tensor-core decode GEMMs: schedule, weight prefixes, fp16 lookup tables, the decode's
// bias, layer-major int16 codes of L layers, feature operand tiles; every segment rounded up to 1 KB.  The codes come
// before the feature tiles so that their place does not depend on F: rqae_intensity_again_f16 reuses them.
struct GemmLayout {
  int L, NKB, F_tiles;
  long long T_pad;
  size_t off_sched, off_wcum, off_lut, off_bias, off_codes, off_u, total;
  long long units() const { return (T_pad / rq::IT_TOK) * (long long)((F_tiles + 1) / 2); }
};

GemmLayout gemm_layout(int L, int nkb, int F, int64_t n_tokens, bool bias) {
  GemmLayout o;
  o.L = L;
  o.NKB = nkb;
  o.F_tiles = (F + rq::IT_FT - 1) / rq::IT_FT;
  o.T_pad = (n_tokens + rq::IT_TOK - 1) / rq::IT_TOK * rq::IT_TOK;
  auto up = [](size_t v) { return (v + 1023) / 1024 * 1024; };
  size_t off = 0;
  o.off_sched = off; off = up(off + (size_t)rq::IT_MAX_KB * sizeof(rq::IntKBlock));
  o.off_wcum = off;  off = up(off + 2 * (size_t)rq::IT_MAX_CUTS * 4);
  o.off_lut = off;   off = up(off + 2 * (size_t)rq::IT_LUT_ROWS * 8);
  o.off_bias = off;  off = up(off + (bias ? (size_t)o.F_tiles * rq::IT_FT * 4 : 0));
  o.off_codes = off; off = up(off + (size_t)L * (size_t)o.T_pad * 2);
  o.off_u = off;     off = up(off + (size_t)o.F_tiles * nkb * rq::IT_U_TILE);
  o.total = off;
  return o;
}

// Runs the GEMM on min(units, sms) persistent CTAs.  Only the intensity epilogue stores through a tensor map; the
// others are given a zeroed one.
template <int EPI>
int launch_gemm(const rq::IntParams& ip, long long units, int sms, const CUtensorMap* out_map, cudaStream_t st) {
  constexpr int smem = rq::IntSmemOf<EPI>::type::TOTAL;
  auto kern = rq::rq_intensity_kernel<EPI>;
  RQ_CUDA(ensure_func_attr((const void*)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  CUtensorMap map;
  if (out_map) map = *out_map;
  else memset(&map, 0, sizeof(map));
  const int grid = (int)(units < sms ? units : sms);
  kern<<<grid, rq::IT_THREADS, smem, st>>>(ip, map);
  RQ_CUDA(launched());
  return RQAE_OK;
}

}  // namespace

extern "C" {

const char* rqae_version(void) { return "rqae_b200 0.1.0 sm_100a"; }

const char* rqae_strerror(int code) {
  switch (code) {
    case RQAE_OK: return "ok";
    case RQAE_EINVAL: return "invalid argument";
    case RQAE_EUNSUPPORTED: return "unsupported shape (codebook_dim must be 4, dim <= 3584, K <= 65535; intensity and tensor-core decode: K < 640, <= 64 cuts; selection: top_k <= 256)";
    case RQAE_ECUDA: return "CUDA runtime error";
    case RQAE_ENODEVICE: return "current device is not an sm_100 (B200) GPU";
    case RQAE_ESIZE: return "buffer too small";
    default: return "unknown error";
  }
}

const char* rqae_last_cuda_error(void) { return cudaGetErrorString(g_last_cuda); }

int64_t rqae_launch_count(int reset) {
  const int64_t v = g_launches;
  if (reset) g_launches = 0;
  return v;
}

size_t rqae_packed_bytes(int nq, int dim, int codebook_dim, int K) {
  RqShape s;
  if (nq <= 0 || dim <= 0 || codebook_dim != 4 || K <= 0 || K > 65535 || rq_pick_shape(dim, &s)) return 0;
  RqLayout L;
  rq_layout(nq, K, &s, &L);
  return L.total;
}

int rqae_pack_weights(const float* w_in, const float* b_in, const float* w_out, const float* b_out,
                      const float* codebook, int codebook_shared, int nq, int dim, int codebook_dim, int K,
                      void* packed, size_t packed_bytes, void* stream) {
  if (!w_in || !b_in || !w_out || !b_out || !codebook || !packed || nq <= 0 || dim <= 0 || K <= 0) return RQAE_EINVAL;
  RqShape s;
  if (codebook_dim != 4 || K > 65535 || rq_pick_shape(dim, &s)) return RQAE_EUNSUPPORTED;
  RqLayout L;
  rq_layout(nq, K, &s, &L);
  if (packed_bytes < L.total) return RQAE_ESIZE;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* pk = (unsigned char*)packed;
  RQ_CUDA(cudaMemsetAsync(pk, 0, RQ_HDR_BYTES, st));
  const long long total = (long long)(nq + 1) * s.E * RQ_GROUP_THREADS;
  pack_stages_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(w_in, b_in, w_out, b_out, nq, dim, s.E, s.CH, pk,
                                                                      L.off_bin, L.off_stage, L.stage_bytes);
  RQ_CUDA(launched());
  if (L.off_stage_cl) {   // second copy for the D-split cluster variant: one chunk per CTA of the cluster
    pack_stages_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(w_in, b_in, w_out, b_out, nq, dim, s.E,
                                                                        rq_cluster_size(s.E), pk, L.off_bin, L.off_stage_cl,
                                                                        L.stage_bytes);
    RQ_CUDA(launched());
  }
  if (codebook_shared) {
    // the table is tiny: fetch it, build the search tables on the host, upload (this entry point therefore
    // synchronises `stream`; it runs once per weight load, never on the hot path)
    std::vector<float> cb_host((size_t)K * 4);
    RQ_CUDA(cudaMemcpyAsync(cb_host.data(), codebook, (size_t)K * 16, cudaMemcpyDeviceToHost, st));
    RQ_CUDA(cudaStreamSynchronize(st));
    SearchTables T;
    build_search_tables(cb_host.data(), K, L.KT, &T);
    RQ_CUDA(cudaMemcpyAsync(pk, &T.hdr, sizeof(T.hdr), cudaMemcpyHostToDevice, st));
    RQ_CUDA(cudaMemcpyAsync(pk + L.off_cbt, T.cbt.data(), T.cbt.size() * 4, cudaMemcpyHostToDevice, st));
    RQ_CUDA(cudaMemcpyAsync(pk + L.off_map, T.map.data(), T.map.size() * 2, cudaMemcpyHostToDevice, st));
    RQ_CUDA(cudaMemcpyAsync(pk + L.off_tp, T.tp.data(), T.tp.size() * 4, cudaMemcpyHostToDevice, st));
    RQ_CUDA(cudaMemcpyAsync(pk + L.off_map3, T.map3.data(), T.map3.size() * 2, cudaMemcpyHostToDevice, st));
    RQ_CUDA(cudaStreamSynchronize(st));
  }
  return RQAE_OK;
}

static void forward_variant_init() {
  if (g_forward_variant.load() < 0) {
    const char* e = getenv("RQAE_CLUSTER");
    g_forward_variant.store(e && atoi(e) != 0 ? 1 : 0);
  }
}

static int forward_common(const void* packed, const float* codebook, int codebook_shared, int nq, int nq_run, int dim,
                          int codebook_dim, int K, int64_t n_tokens, void* codes, int code_dtype, int64_t code_stride,
                          rq::FwdParams& prm, void* stream) {
  if (!packed || !codebook || nq <= 0 || nq_run <= 0 || nq_run > nq || dim <= 0 || K <= 0 || n_tokens < 0) return RQAE_EINVAL;
  if (code_dtype < 0 || code_dtype > 2 || (codes && code_stride < nq_run)) return RQAE_EINVAL;
  if (codes && code_dtype == RQAE_CODE_I16 && K > 32768) return RQAE_EINVAL;   // int16 cannot hold codes >= 32768
  RqShape s;
  if (codebook_dim != 4 || K > 65535 || rq_pick_shape(dim, &s)) return RQAE_EUNSUPPORTED;
  if (n_tokens == 0) return RQAE_OK;
  forward_variant_init();
  int sms = 0;
  int rc = device_sm_count(&sms);
  if (rc) return rc;
  RqLayout L;
  rq_layout(nq, K, &s, &L);
  prm.packed = (const unsigned char*)packed;
  prm.off_bin = L.off_bin; prm.off_cbt = L.off_cbt; prm.off_map = L.off_map; prm.off_stage = L.off_stage;
  prm.off_tp = L.off_tp; prm.off_map3 = L.off_map3;
  prm.codebook = codebook; prm.cb_shared = codebook_shared ? 1 : 0; prm.K = K; prm.nq_run = nq_run; prm.D = dim;
  prm.n_tokens = n_tokens; prm.codes = codes; prm.code_dtype = code_dtype; prm.code_stride = code_stride;
  prm.l2_hot = RQ_L2_HOT_DEFAULT;   // DESIGN.md, "L2 residency of the weight stream"
  cudaStream_t st = (cudaStream_t)stream;
  // Few tokens (the hook's operating point is 4 x 128, scripts/1_create_activations.py:152): units of 2 x 4 tokens
  // instead of 2 x 8 put twice as many SMs to work and halve the time of a pass; a token's arithmetic does not
  // depend on the unit size, so the codes are the same bit for bit.  (Units of 2 x 2 would ask the L2 for more
  // weight bytes per layer than it delivers.)
  const bool few = n_tokens <= (int64_t)sms * 8;
  switch (s.E) {
    case 1: return launch_forward<1, 1, 1, 4, 8>(prm, sms, st);
    case 3: return launch_forward<3, 3, 1, 4, 8>(prm, sms, st);
    case 6: return launch_forward<6, 3, 2, 6, 8>(prm, sms, st);
    case 9:
      if (few) return launch_forward<9, 3, RQ_E9_CH, RQ_E9_NSLOT, 4>(prm, sms, st);
      return launch_forward<9, 3, RQ_E9_CH, RQ_E9_NSLOT, 8>(prm, sms, st);
    case 14: {
      // Gemma-2-9B width, opt-in (rqae_forward_variant(1) / RQAE_CLUSTER=1): the D-split cluster variant -- 2 CTAs x
      // 7 elements per thread, 16 tokens per unit, whole half-stages double-buffered.  Measured (profiles/r2m_*):
      // 302 k tokens/s against 310-318 k of the single-CTA kernel on large batches (the hand-over through the
      // peer's shared memory lengthens the serial chain by what the shorter passes save), 13-43 % faster below
      // ~2400 tokens.  Its summation order differs (c_oracle.KERNEL_ORDER_9B), so it is never chosen silently.
      if (g_forward_variant.load() == 1 && prm.hs == nullptr && L.off_stage_cl) {
        rq::FwdParams pc = prm;
        pc.off_stage = L.off_stage_cl;
        return launch_forward_cluster<7, 7, 1, 2, 8, 2>(pc, sms, st);
      }
      if (few) return launch_forward<14, 2, 7, 10, 4>(prm, sms, st);
      return launch_forward<14, 2, 7, 10, 6>(prm, sms, st);
    }
    default: return RQAE_EUNSUPPORTED;
  }
}

int rqae_forward_f32(const void* packed, const float* codebook, int codebook_shared, int nq, int nq_run, int dim,
                     int codebook_dim, int K, const float* x, int64_t n_tokens, void* codes, int code_dtype,
                     int64_t code_stride, float* q_out, const int32_t* teacher, float* z_out, void* stream) {
  if (n_tokens > 0 && !x) return RQAE_EINVAL;
  rq::FwdParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.x = x; prm.q_out = q_out; prm.teacher = teacher; prm.z_out = z_out;
  return forward_common(packed, codebook, codebook_shared, nq, nq_run, dim, codebook_dim, K, n_tokens, codes, code_dtype,
                        code_stride, prm, stream);
}

int rqae_forward_variant(int variant) {
  forward_variant_init();
  if (variant > 1) return -1;
  const int old = g_forward_variant.load();
  if (variant >= 0) g_forward_variant.store(variant);
  return old;
}

int rqae_hook_rmsnorm(const void* packed, const float* codebook, int codebook_shared, int nq, int nq_run, int dim,
                      int codebook_dim, int K, void* hidden, int hidden_dtype, int64_t n_tokens, int seq_len,
                      const float* rms_weight, float rms_eps, int skip_bos, int replace, void* codes, int code_dtype,
                      int64_t code_stride, void* stream) {
  if (!hidden && n_tokens > 0) return RQAE_EINVAL;
  if (!rms_weight || hidden_dtype < 0 || hidden_dtype > 2 || seq_len <= 0 || !(rms_eps >= 0.0f)) return RQAE_EINVAL;
  rq::FwdParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.hs = hidden; prm.hs_out = replace ? hidden : nullptr; prm.hs_dtype = hidden_dtype; prm.rms_w = rms_weight;
  prm.rms_eps = rms_eps; prm.seq_len = seq_len; prm.skip_bos = skip_bos ? 1 : 0;
  return forward_common(packed, codebook, codebook_shared, nq, nq_run, dim, codebook_dim, K, n_tokens, codes, code_dtype,
                        code_stride, prm, stream);
}

int rqae_decode_f32(const void* packed, const float* codebook0, int nq, int nq_codes, int dim, int codebook_dim, int K,
                    const void* codes, int code_dtype, int64_t code_stride, const float* cv,
                    const uint8_t* layer_mask, int64_t n_tokens, float* q_out, void* stream) {
  if (!packed || !q_out || nq <= 0 || nq_codes < 0 || nq_codes > nq || dim <= 0 || K <= 0 || n_tokens < 0) return RQAE_EINVAL;
  if (!codes && !cv) return RQAE_EINVAL;
  if (codes && (!codebook0 || code_dtype < 0 || code_dtype > 2 || code_stride < nq_codes)) return RQAE_EINVAL;
  RqShape s;
  if (codebook_dim != 4 || K > 65535 || rq_pick_shape(dim, &s)) return RQAE_EUNSUPPORTED;
  if (n_tokens == 0) return RQAE_OK;
  int sms = 0;
  int rc = device_sm_count(&sms);
  if (rc) return rc;
  RqLayout L;
  rq_layout(nq, K, &s, &L);
  rq::DecParams prm;
  prm.packed = (const unsigned char*)packed;
  prm.off_stage = L.off_stage; prm.stage_bytes = L.stage_bytes;
  prm.codebook0 = codebook0; prm.K = K; prm.nq_codes = nq_codes; prm.D = dim; prm.E = s.E; prm.CH = s.CH;
  prm.codes = codes; prm.code_dtype = code_dtype; prm.code_stride = code_stride; prm.cv = cv;
  prm.layer_mask = layer_mask; prm.n_tokens = n_tokens; prm.q_out = q_out;
  rc = rq::launch_decode(prm, sms, (cudaStream_t)stream);
  if (rc == 0) g_launches++;
  if (rc == RQAE_ECUDA) g_last_cuda = cudaGetLastError();
  return rc;
}

int rqae_fp32_peak_probe(int packed_f32x2, int iters, double* flops_per_launch, float* sink, void* stream) {
  if (iters <= 0 || !sink) return RQAE_EINVAL;
  int sms = 0;
  int rc = device_sm_count(&sms);
  if (rc) return rc;
  if (packed_f32x2 >= 2) {   // operand-pattern probes (see fma_pattern_probe_kernel); sink doubles as the data source
    if (packed_f32x2 == 2) fma_pattern_probe_kernel<2><<<sms, 256, 0, (cudaStream_t)stream>>>(iters, sink, sink + 64);
    else fma_pattern_probe_kernel<3><<<sms, 256, 0, (cudaStream_t)stream>>>(iters, sink, sink + 64);
    RQ_CUDA(launched());
    if (flops_per_launch) *flops_per_launch = (double)sms * 256 * (double)iters * (packed_f32x2 == 2 ? 48.0 : 60.0) * 4.0;
    return RQAE_OK;
  }
  const int grid = sms * 2, block = 512;
  if (packed_f32x2) fp32_probe_kernel<true><<<grid, block, 0, (cudaStream_t)stream>>>(iters, sink);
  else fp32_probe_kernel<false><<<grid, block, 0, (cudaStream_t)stream>>>(iters, sink);
  RQ_CUDA(launched());
  if (flops_per_launch) *flops_per_launch = (double)grid * block * (double)iters * 8.0 * 24.0 * 2.0;
  return RQAE_OK;
}

// ---------------------------------------------------------------------------------------------
// host-buffer front end (the end-to-end path)
// ---------------------------------------------------------------------------------------------
// Pipeline options (rqae_forward_host_config; environment defaults RQAE_HOST_CODES = auto|narrow|direct,
// RQAE_HOST_THREADS = n).  Two ways to deliver int32 / int64 codes to a host tensor:
//   narrow  the kernel emits int16 (every code is < K <= 32767), a quarter of the int64 bytes cross PCIe into a
//           pinned staging buffer, and a pool of host threads widens them into the caller's tensor with streaming
//           stores while the next chunk is in flight.  Least PCIe traffic: 11.3 KB per token device -> host.
//   direct  the kernel emits the caller's dtype and the D2H copy lands in the caller's tensor.  No host threads,
//           no staging; 17.4 KB per token device -> host for int64.
// `auto` = narrow.  Measured with one rank per GPU on an 8 x B200 host (tools/e2e_probe.py, profiles/r2c_*): the
// ranks share a host I/O fabric that delivers 185 GB/s host -> device alone, 90 GB/s device -> host alone and
// 64 + 64 GB/s when both directions run, so at 8 ranks the end-to-end rate is bounded by the device -> host
// bytes per token, not by the host cores (one AVX2 widening thread does 1.9 G codes/s; a rank needs 1.2):
// narrow 617 k tokens/s per rank against 549 k direct.  With one or two ranks the two modes tie.
static std::atomic<int> g_host_code_transfer{-1};   // -1: not initialised; 0 auto, 1 narrow, 2 direct
static std::atomic<int> g_host_threads{-1};         // -1: not initialised; 0 auto

static void host_config_init() {
  if (g_host_code_transfer.load() < 0) {
    const char* e = getenv("RQAE_HOST_CODES");
    int v = 0;
    if (e && !strcmp(e, "narrow")) v = 1;
    else if (e && !strcmp(e, "direct")) v = 2;
    g_host_code_transfer.store(v);
  }
  if (g_host_threads.load() < 0) {
    const char* e = getenv("RQAE_HOST_THREADS");
    const int v = e ? atoi(e) : 0;
    g_host_threads.store(v < 0 ? 0 : (v > 64 ? 64 : v));
  }
}

// Widening threads per rank when not given: the host's cores are shared by all ranks of the node
// (LOCAL_WORLD_SIZE, set by torchrun), and half of a rank's share is left to the framework's own threads.
static int host_auto_threads() {
  unsigned hw = std::thread::hardware_concurrency();
  if (hw == 0) hw = 1;
  int lws = 1;
  if (const char* e = getenv("LOCAL_WORLD_SIZE")) lws = atoi(e) > 0 ? atoi(e) : 1;
  int t = (int)hw / (2 * lws);
  return t < 1 ? 1 : (t > 8 ? 8 : t);
}

// int16 -> int32 / int64.  The wide result is written once and not read again by this library: streaming stores
// keep it out of the caches and spare the read-for-ownership of every destination line.
static void widen_range_scalar(const int16_t* src, void* dst, size_t lo, size_t hi, int code_dtype) {
#if defined(__x86_64__) && !defined(RQ_NO_STREAM)
  if (code_dtype == 2) { long long* d = (long long*)dst; for (size_t i = lo; i < hi; i++) _mm_stream_si64(d + i, (long long)src[i]); }
  else { int* d = (int*)dst; for (size_t i = lo; i < hi; i++) _mm_stream_si32(d + i, (int)src[i]); }
  _mm_sfence();
#else
  if (code_dtype == 2) { int64_t* d = (int64_t*)dst; for (size_t i = lo; i < hi; i++) d[i] = src[i]; }
  else { int32_t* d = (int32_t*)dst; for (size_t i = lo; i < hi; i++) d[i] = src[i]; }
#endif
}

#if defined(__x86_64__) && !defined(RQ_NO_STREAM)
__attribute__((target("avx2"))) static void widen_range_avx2(const int16_t* src, void* dst, size_t lo, size_t hi, int code_dtype) {
  size_t i = lo;
  if (code_dtype == 2) {
    long long* d = (long long*)dst;
    for (; i < hi && ((uintptr_t)(d + i) & 31); i++) d[i] = src[i];
    for (; i + 16 <= hi; i += 16) {
      const __m128i a = _mm_loadu_si128((const __m128i*)(src + i));
      const __m128i b = _mm_loadu_si128((const __m128i*)(src + i + 8));
      _mm256_stream_si256((__m256i*)(d + i), _mm256_cvtepi16_epi64(a));
      _mm256_stream_si256((__m256i*)(d + i + 4), _mm256_cvtepi16_epi64(_mm_srli_si128(a, 8)));
      _mm256_stream_si256((__m256i*)(d + i + 8), _mm256_cvtepi16_epi64(b));
      _mm256_stream_si256((__m256i*)(d + i + 12), _mm256_cvtepi16_epi64(_mm_srli_si128(b, 8)));
    }
    for (; i < hi; i++) d[i] = src[i];
  } else {
    int* d = (int*)dst;
    for (; i < hi && ((uintptr_t)(d + i) & 31); i++) d[i] = src[i];
    for (; i + 16 <= hi; i += 16) {
      const __m128i a = _mm_loadu_si128((const __m128i*)(src + i));
      const __m128i b = _mm_loadu_si128((const __m128i*)(src + i + 8));
      _mm256_stream_si256((__m256i*)(d + i), _mm256_cvtepi16_epi32(a));
      _mm256_stream_si256((__m256i*)(d + i + 8), _mm256_cvtepi16_epi32(b));
    }
    for (; i < hi; i++) d[i] = src[i];
  }
  _mm_sfence();
}
#endif

static void widen_range(const int16_t* src, void* dst, size_t lo, size_t hi, int code_dtype) {
#if defined(__x86_64__) && !defined(RQ_NO_STREAM)
  static const bool avx2 = __builtin_cpu_supports("avx2");
  if (avx2) { widen_range_avx2(src, dst, lo, hi, code_dtype); return; }
#endif
  widen_range_scalar(src, dst, lo, hi, code_dtype);
}

// Persistent worker pool of the calling thread's pipeline (the first version spawned threads per chunk).
class WidenPool {
 public:
  ~WidenPool() { stop(); }
  void resize(int workers) {
    if ((int)th_.size() == workers) return;
    stop();
    stop_ = false;
    const unsigned long long g0 = gen_;   // a new worker must not mistake an old generation for a job
    for (int i = 0; i < workers; i++) th_.emplace_back([this, i, g0] { loop(i + 1, g0); });
  }
  int workers() const { return (int)th_.size(); }
  // splits [0, n) over the workers and the caller; returns when all parts are done
  void run(const int16_t* src, void* dst, size_t n, int code_dtype) {
    const int parts = (int)th_.size() + 1;
    if (parts == 1 || n < (1u << 16)) { widen_range(src, dst, 0, n, code_dtype); return; }
    {
      std::lock_guard<std::mutex> lk(mu_);
      src_ = src; dst_ = dst; n_ = n; dtype_ = code_dtype; parts_ = parts;
      pending_ = (int)th_.size();
      gen_++;
    }
    go_.notify_all();
    part(0);
    std::unique_lock<std::mutex> lk(mu_);
    done_.wait(lk, [this] { return pending_ == 0; });
  }

 private:
  void part(int id) {
    const size_t per = ((n_ + parts_ - 1) / parts_ + 15) & ~(size_t)15;
    const size_t lo = per * id, hi = lo + per < n_ ? lo + per : n_;
    if (lo < hi) widen_range(src_, dst_, lo, hi, dtype_);
  }
  void loop(int id, unsigned long long seen) {
    for (;;) {
      {
        std::unique_lock<std::mutex> lk(mu_);
        go_.wait(lk, [&] { return stop_ || gen_ != seen; });
        if (stop_) return;
        seen = gen_;
      }
      part(id);
      std::lock_guard<std::mutex> lk(mu_);
      if (--pending_ == 0) done_.notify_one();
    }
  }
  void stop() {
    {
      std::lock_guard<std::mutex> lk(mu_);
      stop_ = true;
    }
    go_.notify_all();
    for (auto& t : th_) t.join();
    th_.clear();
  }
  std::vector<std::thread> th_;
  std::mutex mu_;
  std::condition_variable go_, done_;
  unsigned long long gen_ = 0;
  int pending_ = 0, parts_ = 1, dtype_ = 2;
  bool stop_ = false;
  const int16_t* src_ = nullptr;
  void* dst_ = nullptr;
  size_t n_ = 0;
};

// Cached resources of the host pipeline (per calling thread): device staging buffers, a pinned staging
// area for narrow codes, streams and events.  Re-created when a call needs more room or another device.
constexpr int kHostBufs = 3;
struct HostPipe {
  int dev = -1;
  size_t x_bytes = 0, q_bytes = 0, c_bytes = 0, h_bytes = 0;
  float* dx[kHostBufs] = {};
  float* dq[kHostBufs] = {};
  void* dc[kHostBufs] = {};
  void* hc[kHostBufs] = {};   // pinned
  cudaStream_t s_in = nullptr, s_cmp = nullptr, s_out = nullptr;
  cudaEvent_t ev_in[kHostBufs] = {}, ev_cmp[kHostBufs] = {}, ev_out[kHostBufs] = {};
  WidenPool pool;
  void release() {
    for (int b = 0; b < kHostBufs; b++) {
      if (dx[b]) cudaFree(dx[b]);
      if (dq[b]) cudaFree(dq[b]);
      if (dc[b]) cudaFree(dc[b]);
      if (hc[b]) cudaFreeHost(hc[b]);
      if (ev_in[b]) cudaEventDestroy(ev_in[b]);
      if (ev_cmp[b]) cudaEventDestroy(ev_cmp[b]);
      if (ev_out[b]) cudaEventDestroy(ev_out[b]);
      dx[b] = dq[b] = nullptr; dc[b] = hc[b] = nullptr; ev_in[b] = ev_cmp[b] = ev_out[b] = nullptr;
    }
    if (s_in) cudaStreamDestroy(s_in);
    if (s_cmp) cudaStreamDestroy(s_cmp);
    if (s_out) cudaStreamDestroy(s_out);
    s_in = s_cmp = s_out = nullptr;
    x_bytes = q_bytes = c_bytes = h_bytes = 0;
    dev = -1;
  }
};
static thread_local HostPipe g_pipe;

int rqae_forward_host_release(void) {
  g_pipe.release();
  g_pipe.pool.resize(0);
  return RQAE_OK;
}

int rqae_widen_codes_host(const int16_t* src_host, void* dst_host, int64_t n, int code_dtype, int threads) {
  if ((!src_host || !dst_host) && n > 0) return RQAE_EINVAL;
  if (n < 0 || (code_dtype != RQAE_CODE_I32 && code_dtype != RQAE_CODE_I64) || threads < 0 || threads > 64) return RQAE_EINVAL;
  static thread_local WidenPool pool;
  pool.resize((threads > 0 ? threads : host_auto_threads()) - 1);
  pool.run(src_host, dst_host, (size_t)n, code_dtype);
  return RQAE_OK;
}

int rqae_forward_host_config(int code_transfer, int widen_threads) {
  host_config_init();
  if (code_transfer > 2 || widen_threads > 64) return RQAE_EINVAL;
  if (code_transfer >= 0) g_host_code_transfer.store(code_transfer);
  if (widen_threads >= 0) g_host_threads.store(widen_threads);
  return RQAE_OK;
}

int rqae_forward_host_mode(int* code_transfer, int* widen_threads) {
  host_config_init();
  if (code_transfer) *code_transfer = g_host_code_transfer.load() == 2 ? 2 : 1;
  if (widen_threads) *widen_threads = g_host_threads.load() > 0 ? g_host_threads.load() : host_auto_threads();
  return RQAE_OK;
}

int rqae_forward_host_f32(const void* packed, const float* codebook, int codebook_shared, int nq, int nq_run, int dim,
                          int codebook_dim, int K, const float* x_host, int64_t n_tokens, void* codes_host,
                          int code_dtype, float* q_host, int64_t chunk_tokens) {
  if (!packed || !codebook || !x_host || n_tokens < 0 || chunk_tokens <= 0 || code_dtype < 0 || code_dtype > 2) return RQAE_EINVAL;
  if (nq_run <= 0 || nq_run > nq) return RQAE_EINVAL;
  if (code_dtype == RQAE_CODE_I16 && K > 32768) return RQAE_EINVAL;   // int16 cannot hold the codes
  if (n_tokens == 0) return RQAE_OK;
  if (chunk_tokens > n_tokens) chunk_tokens = n_tokens;
  host_config_init();
  const int mode = g_host_code_transfer.load();
  const bool narrow = codes_host != nullptr && code_dtype != RQAE_CODE_I16 && K <= 32767 && mode != 2;
  const int dev_dtype = narrow ? RQAE_CODE_I16 : code_dtype;
  const size_t dsz = dev_dtype == 2 ? 8 : (dev_dtype == 1 ? 4 : 2);     // code size on the device / on the wire
  const size_t usz = code_dtype == 2 ? 8 : (code_dtype == 1 ? 4 : 2);   // code size in the caller's tensor

  HostPipe& P = g_pipe;
  int dev = 0;
  RQ_CUDA(cudaGetDevice(&dev));
  const size_t need_x = (size_t)chunk_tokens * dim * 4, need_q = q_host ? need_x : 0;
  const size_t need_c = codes_host ? (size_t)chunk_tokens * nq_run * dsz : 0, need_h = narrow ? need_c : 0;
  if (P.dev != dev || P.x_bytes < need_x || P.q_bytes < need_q || P.c_bytes < need_c || P.h_bytes < need_h) {
    P.release();
    P.dev = dev;
    RQ_CUDA(cudaStreamCreateWithFlags(&P.s_in, cudaStreamNonBlocking));
    RQ_CUDA(cudaStreamCreateWithFlags(&P.s_cmp, cudaStreamNonBlocking));
    RQ_CUDA(cudaStreamCreateWithFlags(&P.s_out, cudaStreamNonBlocking));
    for (int b = 0; b < kHostBufs; b++) {
      RQ_CUDA(cudaMalloc(&P.dx[b], need_x));
      if (need_q) RQ_CUDA(cudaMalloc(&P.dq[b], need_q));
      if (need_c) RQ_CUDA(cudaMalloc(&P.dc[b], need_c));
      if (need_h) RQ_CUDA(cudaHostAlloc(&P.hc[b], need_h, cudaHostAllocDefault));
      RQ_CUDA(cudaEventCreateWithFlags(&P.ev_in[b], cudaEventDisableTiming));
      RQ_CUDA(cudaEventCreateWithFlags(&P.ev_cmp[b], cudaEventDisableTiming));
      RQ_CUDA(cudaEventCreateWithFlags(&P.ev_out[b], cudaEventDisableTiming));
    }
    P.x_bytes = need_x; P.q_bytes = need_q; P.c_bytes = need_c; P.h_bytes = need_h;
  }
  if (narrow) {
    const int t = g_host_threads.load() > 0 ? g_host_threads.load() : host_auto_threads();
    P.pool.resize(t - 1);   // the calling thread is one of them
  }

  int rc = RQAE_OK;
  cudaError_t err = cudaSuccess;
#define RQ_TRY(call)                                        \
  do {                                                      \
    if (rc == RQAE_OK && err == cudaSuccess) err = (call);  \
  } while (0)
  const int64_t n_chunks = (n_tokens + chunk_tokens - 1) / chunk_tokens;
  auto chunk_len = [&](int64_t c) { const int64_t t0 = c * chunk_tokens; return (n_tokens - t0 < chunk_tokens) ? (n_tokens - t0) : chunk_tokens; };
  auto finish_chunk = [&](int64_t c) {   // host side of chunk c: wait for its D2H copies, widen the codes
    const int b = (int)(c % kHostBufs);
    RQ_TRY(cudaEventSynchronize(P.ev_out[b]));
    if (rc == RQAE_OK && err == cudaSuccess)
      P.pool.run((const int16_t*)P.hc[b], (char*)codes_host + (size_t)c * chunk_tokens * nq_run * usz,
                 (size_t)chunk_len(c) * nq_run, code_dtype);
  };
  for (int64_t c = 0; c < n_chunks && rc == RQAE_OK && err == cudaSuccess; c++) {
    const int b = (int)(c % kHostBufs);
    const int64_t t0 = c * chunk_tokens;
    const int64_t nt = chunk_len(c);
    // buffer set b was last used by chunk c - kHostBufs: its input is free once that kernel has run, its outputs
    // once their D2H copies are done -- and, in narrow mode, once the host has widened the staged codes, which
    // finish_chunk(c - kHostBufs) did before this iteration (it runs kHostBufs - 1 chunks behind the enqueue)
    if (c >= kHostBufs) RQ_TRY(cudaStreamWaitEvent(P.s_in, P.ev_cmp[b], 0));
    RQ_TRY(cudaMemcpyAsync(P.dx[b], x_host + (size_t)t0 * dim, (size_t)nt * dim * 4, cudaMemcpyHostToDevice, P.s_in));
    RQ_TRY(cudaEventRecord(P.ev_in[b], P.s_in));
    RQ_TRY(cudaStreamWaitEvent(P.s_cmp, P.ev_in[b], 0));
    if (c >= kHostBufs) RQ_TRY(cudaStreamWaitEvent(P.s_cmp, P.ev_out[b], 0));
    if (err != cudaSuccess) break;
    rc = rqae_forward_f32(packed, codebook, codebook_shared, nq, nq_run, dim, codebook_dim, K, P.dx[b], nt,
                          codes_host ? P.dc[b] : nullptr, dev_dtype, nq_run, q_host ? P.dq[b] : nullptr, nullptr, nullptr,
                          (void*)P.s_cmp);
    if (rc) break;
    RQ_TRY(cudaEventRecord(P.ev_cmp[b], P.s_cmp));
    RQ_TRY(cudaStreamWaitEvent(P.s_out, P.ev_cmp[b], 0));
    if (codes_host) {
      void* dst = narrow ? P.hc[b] : (void*)((char*)codes_host + (size_t)t0 * nq_run * usz);
      RQ_TRY(cudaMemcpyAsync(dst, P.dc[b], (size_t)nt * nq_run * dsz, cudaMemcpyDeviceToHost, P.s_out));
    }
    if (q_host) RQ_TRY(cudaMemcpyAsync(q_host + (size_t)t0 * dim, P.dq[b], (size_t)nt * dim * 4, cudaMemcpyDeviceToHost, P.s_out));
    RQ_TRY(cudaEventRecord(P.ev_out[b], P.s_out));
    // chunk c is queued; while the GPU works on it, finish an earlier chunk on the host.  Its staging buffer is
    // reused by chunk c + 1, which is enqueued only after this returns.
    if (narrow && c >= kHostBufs - 1) finish_chunk(c - (kHostBufs - 1));
  }
  if (narrow)
    for (int64_t c = (n_chunks > kHostBufs - 1 ? n_chunks - (kHostBufs - 1) : 0); c < n_chunks; c++) finish_chunk(c);
#undef RQ_TRY
  // drain every stream even after a failure: the buffers may be re-used by the next call
  const cudaError_t e1 = cudaStreamSynchronize(P.s_in), e2 = cudaStreamSynchronize(P.s_cmp), e3 = cudaStreamSynchronize(P.s_out);
  if (err == cudaSuccess) err = e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3);
  if (rc == RQAE_OK && err != cudaSuccess) { g_last_cuda = err; rc = RQAE_ECUDA; }
  return rc;
}

// ---------------------------------------------------------------------------------------------
// feature intensities (rq_intensity.cuh)
// ---------------------------------------------------------------------------------------------
// 3-D tensor map of the intensity output out[f][cut][t] (fp16) for the epilogue's TMA stores: box = 32 features x 1 cut
// x 64 tokens, 128-byte swizzle.  cuTensorMapEncodeTiled is a driver entry point; it is looked up through the runtime
// so that the library does not link against libcuda.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static int make_out_map(void* out, int64_t out_stride, int n_cuts, int n_features, CUtensorMap* map) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    const cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !f) { g_last_cuda = e != cudaSuccess ? e : cudaErrorSymbolNotFound; return RQAE_ECUDA; }
    fn = (EncodeTiledFn)f;
  }
  const cuuint64_t gdim[3] = {(cuuint64_t)out_stride, (cuuint64_t)n_cuts, (cuuint64_t)n_features};
  const cuuint64_t gstride[2] = {(cuuint64_t)out_stride * 2, (cuuint64_t)out_stride * 2 * (cuuint64_t)n_cuts};
  const cuuint32_t box[3] = {64, 1, 32};
  const cuuint32_t estride[3] = {1, 1, 1};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, out, gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { g_last_cuda = cudaErrorInvalidValue; return RQAE_ECUDA; }
  return RQAE_OK;
}

// The intensity workspace for a list of cuts (strictly ascending layer indices).
static int int_layout(const int32_t* cuts, int n_cuts, int F, int64_t n_tokens, GemmLayout* o) {
  if (!cuts || n_cuts <= 0 || n_cuts > rq::IT_MAX_CUTS || F <= 0 || n_tokens < 0) return RQAE_EINVAL;
  int prev = -1, nkb = 0;
  for (int c = 0; c < n_cuts; c++) {
    if (cuts[c] <= prev) return RQAE_EINVAL;   // strictly ascending layer indices
    nkb += (cuts[c] - prev + rq::IT_LPB - 1) / rq::IT_LPB;
    prev = cuts[c];
  }
  if (nkb > rq::IT_MAX_KB) return RQAE_EUNSUPPORTED;
  *o = gemm_layout(prev + 1, nkb, F, n_tokens, false);
  return RQAE_OK;
}

size_t rqae_intensity_workspace_bytes(const int32_t* cuts_host, int n_cuts, int n_features, int64_t n_tokens) {
  GemmLayout L;
  if (int_layout(cuts_host, n_cuts, n_features, n_tokens, &L)) return 0;
  return L.total;
}

static int intensity_impl(const float* cb_norm, int K, const void* codes, int code_dtype, int64_t code_stride,
                          int64_t n_tokens, const int32_t* centers, int64_t center_stride, int n_features,
                          const void* layer_weights_f16, const int32_t* cuts_host, int n_cuts, void* out,
                          int64_t out_stride, void* workspace, size_t workspace_bytes, void* stream, bool reuse_codes);

int rqae_intensity_f16(const float* cb_norm, int K, const void* codes, int code_dtype, int64_t code_stride,
                       int64_t n_tokens, const int32_t* centers, int64_t center_stride, int n_features,
                       const void* layer_weights_f16, const int32_t* cuts_host, int n_cuts, void* out,
                       int64_t out_stride, void* workspace, size_t workspace_bytes, void* stream) {
  if (!codes) return RQAE_EINVAL;
  return intensity_impl(cb_norm, K, codes, code_dtype, code_stride, n_tokens, centers, center_stride, n_features, layer_weights_f16,
                        cuts_host, n_cuts, out, out_stride, workspace, workspace_bytes, stream, false);
}

int rqae_intensity_again_f16(const float* cb_norm, int K, int64_t n_tokens, const int32_t* centers, int64_t center_stride,
                             int n_features, const void* layer_weights_f16, const int32_t* cuts_host, int n_cuts, void* out,
                             int64_t out_stride, void* workspace, size_t workspace_bytes, void* stream) {
  return intensity_impl(cb_norm, K, nullptr, 0, 1 << 30, n_tokens, centers, center_stride, n_features, layer_weights_f16, cuts_host,
                        n_cuts, out, out_stride, workspace, workspace_bytes, stream, true);
}

static int intensity_impl(const float* cb_norm, int K, const void* codes, int code_dtype, int64_t code_stride,
                          int64_t n_tokens, const int32_t* centers, int64_t center_stride, int n_features,
                          const void* layer_weights_f16, const int32_t* cuts_host, int n_cuts, void* out,
                          int64_t out_stride, void* workspace, size_t workspace_bytes, void* stream, bool reuse_codes) {
  if (!cb_norm || (!codes && !reuse_codes) || !centers || !layer_weights_f16 || !out || !workspace || K <= 0) return RQAE_EINVAL;
  if (code_dtype < 0 || code_dtype > 2) return RQAE_EINVAL;
  if (K + 1 > rq::IT_LUT_ROWS) return RQAE_EUNSUPPORTED;
  GemmLayout L;
  int rc = int_layout(cuts_host, n_cuts, n_features, n_tokens, &L);
  if (rc) return rc;
  if (code_stride < L.L || center_stride < L.L) return RQAE_EINVAL;
  if (out_stride < L.T_pad || (out_stride & 7) || ((uintptr_t)out & 15)) return RQAE_EINVAL;   // 16-byte row stores of 256 tokens
  if (((uintptr_t)workspace & 1023) || workspace_bytes < L.total) return RQAE_ESIZE;
  if (n_tokens == 0) return RQAE_OK;
  int sms = 0;
  rc = device_sm_count(&sms);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* ws = (unsigned char*)workspace;
  // 1. schedule, weight prefixes, fp16 lookup table
  rq::IntPrepParams pp;
  memset(&pp, 0, sizeof(pp));
  for (int c = 0; c < n_cuts; c++) pp.cuts[c] = cuts_host[c];
  pp.n_cuts = n_cuts; pp.K = K; pp.cb_norm = cb_norm; pp.w = (const __half*)layer_weights_f16;
  pp.sched = (rq::IntKBlock*)(ws + L.off_sched); pp.wcum = (float*)(ws + L.off_wcum); pp.lut = (uint2*)(ws + L.off_lut);
  rq::int_prep_kernel<<<4, 256, 0, st>>>(pp);
  RQ_CUDA(launched());
  // 2. codes -> layer-major int16 (kept from the previous call on this workspace when the caller says they are the same)
  if (!reuse_codes) {
    dim3 grid((unsigned)(L.T_pad / rq::IT_TOK), (unsigned)((L.L + 31) / 32)), block(256);
    uint32_t* ct = (uint32_t*)(ws + L.off_codes);
    with_code_type(code_dtype, [&](auto tag) {
      using CT = decltype(tag);
      rq::int_transpose_kernel<CT><<<grid, block, 0, st>>>((const CT*)codes, code_stride, n_tokens, L.L, K, false, ct);
    });
    RQ_CUDA(launched());
  }
  // 3. feature operand tiles
  {
    const long long total = (long long)L.F_tiles * L.NKB * rq::IT_FT * rq::IT_LPB;
    rq::int_pack_u_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(
        centers, center_stride, n_features, L.F_tiles, L.NKB, (const rq::IntKBlock*)(ws + L.off_sched), cb_norm, K,
        (const __half*)layer_weights_f16, ws + L.off_u);
    RQ_CUDA(launched());
  }
  // 4. the GEMM
  rq::IntParams ip;
  ip.codes_p = (const uint32_t*)(ws + L.off_codes); ip.L = L.L; ip.T_pad = L.T_pad; ip.u_tiles = ws + L.off_u;
  ip.sched = (const rq::IntKBlock*)(ws + L.off_sched); ip.wcum = (const float*)(ws + L.off_wcum);
  ip.lut = (const uint2*)(ws + L.off_lut); ip.K = K; ip.NKB = L.NKB; ip.n_cuts = n_cuts; ip.F = n_features;
  // start groups 20 k clocks apart when every CTA has several units to run
  ip.stagger = L.units() >= 4LL * sms && n_cuts >= 4 ? 20000 : 0;
  ip.q_out = nullptr; ip.bias = nullptr; ip.T = n_tokens; ip.D = 0;
  ip.F_tiles = L.F_tiles; ip.out = (__half*)out; ip.out_stride = out_stride; ip.n_tok_tiles = L.T_pad / rq::IT_TOK;
  CUtensorMap out_map;
  rc = make_out_map(out, out_stride, n_cuts, n_features, &out_map);
  if (rc) return rc;
  return launch_gemm<0>(ip, L.units(), sms, &out_map, st);
}

int rqae_intensity_exact_f16(const void* sims_f16, int K, const void* codes, int code_dtype, int64_t code_stride,
                             int64_t n_tokens, const int32_t* centers, int64_t center_stride, int n_features,
                             const void* layer_weights_f16, const int32_t* cuts_host, int n_cuts, void* out,
                             int64_t out_stride, void* stream) {
  if (!sims_f16 || !codes || !centers || !layer_weights_f16 || !cuts_host || !out) return RQAE_EINVAL;
  if (K <= 0 || code_dtype < 0 || code_dtype > 2 || n_tokens < 0 || n_features < 0 || n_cuts <= 0) return RQAE_EINVAL;
  if (K >= rq::IX_ROWS) return RQAE_EUNSUPPORTED;   // K + 1 slab rows
  int prev = -1;
  for (int c = 0; c < n_cuts; c++) {
    if (cuts_host[c] <= prev) return RQAE_EINVAL;   // strictly ascending, >= 0
    prev = cuts_host[c];
    if (prev >= rq::IX_MAX_LAYERS) return RQAE_EUNSUPPORTED;
  }
  if (code_stride <= prev || center_stride <= prev) return RQAE_EINVAL;
  if (out_stride < (n_tokens + 7) / 8 * 8 || (out_stride & 7) || ((uintptr_t)out & 15)) return RQAE_EINVAL;   // the selection's rows
  if (n_tokens == 0 || n_features == 0) return RQAE_OK;
  int sms = 0;
  int rc = device_sm_count(&sms);
  if (rc) return rc;
  rq::IxParams xp;
  memset(&xp, 0, sizeof(xp));
  for (int c = 0; c < n_cuts; c++) xp.cut_mask[cuts_host[c] >> 5] |= 1u << (cuts_host[c] & 31);
  xp.sims = (const __half*)sims_f16; xp.codes = codes; xp.code_stride = code_stride; xp.n_tokens = n_tokens;
  xp.n_tiles = (n_tokens + rq::IX_TILE - 1) / rq::IX_TILE; xp.centers = centers; xp.center_stride = center_stride;
  xp.w = (const __half*)layer_weights_f16; xp.out = (__half*)out; xp.out_stride = out_stride;
  xp.K = K; xp.F = n_features; xp.n_groups = (n_features + rq::IX_FG - 1) / rq::IX_FG; xp.n_cuts = n_cuts; xp.L = prev + 1;
  const long long units = xp.n_tiles * xp.n_groups;
  const unsigned grid = (unsigned)std::min<long long>(units, 2LL * sms);   // two CTAs per SM
  cudaError_t e = cudaSuccess;
  with_code_type(code_dtype, [&](auto tag) {
    const void* kern = (const void*)rq::rq_intensity_exact_kernel<decltype(tag)>;
    e = ensure_func_attr(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, rq::IX_SMEM);
    if (e == cudaSuccess) {
      rq::rq_intensity_exact_kernel<decltype(tag)><<<grid, rq::IX_THREADS, rq::IX_SMEM, (cudaStream_t)stream>>>(xp);
      e = launched();
    }
  });
  RQ_CUDA(e);
  return RQAE_OK;
}

int rqae_select_top_middle_bottom_f16(const void* vals, int64_t rows, int64_t row_stride, int64_t n, int top_k,
                                      int32_t* idx_out, void* val_out, void* stream) {
  if (!vals || !idx_out || rows < 0 || top_k < 1 || n < top_k || n >= (int64_t)1 << 31) return RQAE_EINVAL;
  if (top_k > rq::MN_KMAX) return RQAE_EUNSUPPORTED;
  if ((row_stride & 7) || row_stride < (n + 7) / 8 * 8 || ((uintptr_t)vals & 15)) return RQAE_EINVAL;   // 16-byte row loads
  if (rows == 0) return RQAE_OK;
  int sms = 0;
  int rc = device_sm_count(&sms);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  rq::MineParams mp;
  mp.vals = (const __half*)vals; mp.rows = rows; mp.row_stride = row_stride; mp.n = n; mp.k = top_k;
  mp.idx_out = idx_out; mp.val_out = (__half*)val_out;
  // RQAE_MINE_V2=1 keeps the three-pass kernel for every row (A/B timing against the sample-bracketed one)
  const bool v2 = [] { const char* e = getenv("RQAE_MINE_V2"); return e && atoi(e) != 0; }();   // read per call: A/B in one process
  constexpr int smem2 = rq::M2_SMEM_BYTES_PAD + rq::M2_LP_BYTES + (int)sizeof(rq::Mine2Smem);
  constexpr int per_sm2 = 16 / rq::M2_WARPS;
  static_assert(smem2 <= (228 * 1024 - per_sm2 * 1024) / per_sm2, "shared memory budget");
  if (!v2 && n >= 16384 && n <= 262144 && rows < ((int64_t)1 << 31)) {
    // rq_mine3_kernel: brackets from a sample, one streaming pass, exact selection among the candidates; rows whose
    // brackets miss are finished by rq_mine2_kernel in list mode
    const int slog = n <= 131072 ? 4 : 3;
    const double ms = (double)(((n / 16) >> slog) * 16), s = (double)n / ms, sig = 0.5 * sqrt(ms);
    // half-width of the median bracket in sigmas of the sample's rank error (sweep of 4.5 / 4 / 3.5 / 3:
    // profiles/r5z_select_z_sweep.txt)
    constexpr double z = 4.0;
    const long long kh = top_k / 2, m0 = n / 2 - kh, m1 = n / 2 + kh;
    mp.sample_log2 = slog;
    mp.c_top = (int)ceil(top_k / s + 6.0 * sqrt(top_k / s) + 3.0);
    mp.c_hi = (int)floor((double)m0 / s - z * sig) - 1;
    mp.c_lo = (int)ceil((double)m1 / s + z * sig) + 1;
    int* fb = nullptr;
    cudaMemPool_t pool;
    RQ_CUDA(scratch_pool(&pool));
    RQ_CUDA(cudaMallocFromPoolAsync((void**)&fb, (size_t)(rows + 1) * sizeof(int), pool, st));
    cudaError_t e = cudaMemsetAsync(fb, 0, sizeof(int), st);
    if (e == cudaSuccess) {
      mp.fb_count = fb; mp.fb_list = fb + 1;
      constexpr int smem3 = (int)sizeof(rq::Mine3Smem);
      static_assert(2 * (smem3 + 1024) <= 227 * 1024, "two CTAs per SM");
      e = ensure_func_attr((const void*)rq::rq_mine3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem3);
      if (e == cudaSuccess) {
        const int grid = (int)(rows < 2LL * sms ? rows : 2LL * sms);
        rq::rq_mine3_kernel<<<grid, rq::M3_THREADS, smem3, st>>>(mp);
        e = launched();
      }
      if (e == cudaSuccess) e = ensure_func_attr((const void*)rq::rq_mine2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2);
      if (e == cudaSuccess) {
        rq::MineParams fp = mp;
        fp.row_count = fb; fp.row_list = fb + 1;
        const long long cap = (long long)sms * per_sm2;
        rq::rq_mine2_kernel<<<(int)(rows < cap ? rows : cap), rq::M2_THREADS, smem2, st>>>(fp);
        e = launched();
      }
    }
    cudaFreeAsync(fb, st);
    RQ_CUDA(e);
    return RQAE_OK;
  }
  RQ_CUDA(ensure_func_attr((const void*)rq::rq_mine2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2));
  const int grid = (int)(rows < (long long)sms * per_sm2 ? rows : (long long)sms * per_sm2);
  rq::rq_mine2_kernel<<<grid, rq::M2_THREADS, smem2, st>>>(mp);
  RQ_CUDA(launched());
  return RQAE_OK;
}

// ---------------------------------------------------------------------------------------------
// nearest-example search over a code store (rq_search.cuh; demo/server/server.py:159-325)
// ---------------------------------------------------------------------------------------------
size_t rqae_search_table_bytes(int n_layers, int K) {
  if (n_layers <= 0 || K <= 0) return 0;
  return (size_t)n_layers * (size_t)K * rq::SR_Q * sizeof(__half);
}

int rqae_search_build_table_f16(const void* sims_f16, int K, const int32_t* query, int64_t query_stride, int n_query,
                                int n_layers, void* table, size_t table_bytes, void* stream) {
  if (!sims_f16 || !query || !table || K <= 0 || n_layers <= 0 || n_query <= 0 || query_stride < n_layers) return RQAE_EINVAL;
  if (n_query > rq::SR_Q || n_layers > 65535) return RQAE_EUNSUPPORTED;
  if (((uintptr_t)table & 15)) return RQAE_EINVAL;
  if (table_bytes < rqae_search_table_bytes(n_layers, K)) return RQAE_ESIZE;
  int sms = 0;
  int rc = device_sm_count(&sms);
  if (rc) return rc;
  rq::SearchTableParams tp;
  tp.sims = (const __half*)sims_f16; tp.query = query; tp.query_stride = query_stride;
  tp.n_query = n_query; tp.n_layers = n_layers; tp.K = K; tp.table = (__half*)table;
  dim3 grid((unsigned)((K + 31) / 32), (unsigned)n_layers);
  rq::search_table_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(tp);
  RQ_CUDA(launched());
  return RQAE_OK;
}

int rqae_search_accumulate_f16(const void* table, int K, const void* codes, int code_dtype, int64_t code_stride,
                               int64_t n_tokens, int layer_begin, int layer_end, int first, void* acc, void* stream) {
  if (!table || !codes || !acc || K <= 0 || n_tokens < 0) return RQAE_EINVAL;
  if (code_dtype < 0 || code_dtype > 2) return RQAE_EINVAL;
  if (layer_begin < 0 || layer_end <= layer_begin || code_stride < layer_end) return RQAE_EINVAL;
  if (((uintptr_t)table & 7) || ((uintptr_t)acc & 7)) return RQAE_EINVAL;     // 8-byte lane accesses
  if (n_tokens == 0) return RQAE_OK;
  int sms = 0;
  int rc = device_sm_count(&sms);
  if (rc) return rc;
  rq::SearchAccParams ap;
  ap.table = (const __half*)table; ap.codes = codes; ap.code_stride = code_stride; ap.n_tokens = n_tokens;
  ap.K = K; ap.layer_begin = layer_begin; ap.layer_end = layer_end; ap.first = first ? 1 : 0; ap.acc = (__half*)acc;
  const long long tiles = (n_tokens + rq::SR_TILE - 1) / rq::SR_TILE;
  const int grid = (int)(tiles < 4LL * sms ? tiles : 4LL * sms);
  with_code_type(code_dtype, [&](auto tag) {
    rq::search_accumulate_kernel<decltype(tag)><<<grid, rq::SR_THREADS, 0, (cudaStream_t)stream>>>(ap);
  });
  RQ_CUDA(launched());
  return RQAE_OK;
}

int rqae_search_position_max_f16(const void* acc, int64_t n_seq, int seq_len, int n_query, void* out,
                                 int64_t out_stride, void* stream) {
  if (!acc || !out || n_seq < 0 || seq_len <= 0 || n_query <= 0) return RQAE_EINVAL;
  if (n_query > rq::SR_Q) return RQAE_EUNSUPPORTED;
  if (out_stride < n_seq || (out_stride & 7) || ((uintptr_t)out & 15)) return RQAE_EINVAL;   // the layout rqae_select_top_middle_bottom_f16 reads
  if ((uintptr_t)acc & 7) return RQAE_EINVAL;                                                // 8-byte lane loads
  if (out_stride == 0) return RQAE_OK;
  int sms = 0;
  int rc = device_sm_count(&sms);
  if (rc) return rc;
  rq::SearchMaxParams mp;
  mp.acc = (const __half*)acc; mp.n_seq = n_seq; mp.out_stride = out_stride; mp.seq_len = seq_len; mp.n_query = n_query;
  mp.out = (__half*)out;
  const long long blocks = (out_stride + 31) / 32;
  if (blocks >= (1LL << 31)) return RQAE_EUNSUPPORTED;
  rq::search_posmax_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(mp);
  RQ_CUDA(launched());
  return RQAE_OK;
}

// ---------------------------------------------------------------------------------------------
// tensor-core form of the search maxima (opt-in) and the exact rows of the selected sequences
// ---------------------------------------------------------------------------------------------
static int srch_tc_nkb(const int32_t* layers, int n_layers_list, int* nkb_out, int* last_out) {
  if (!layers || n_layers_list <= 0 || n_layers_list > rq::IT_MAX_CUTS) return RQAE_EINVAL;
  int a = 0, nkb = 0;
  for (int c = 0; c < n_layers_list; c++) {
    const int b = layers[c];
    if (b <= a) return RQAE_EINVAL;                    // strictly ascending positive range ends
    nkb += (b - 1) / 8 - a / 8 + 1;
    a = b;
  }
  if (nkb > rq::IT_MAX_KB) return RQAE_EUNSUPPORTED;
  *nkb_out = nkb;
  *last_out = a;
  return RQAE_OK;
}

size_t rqae_search_tc_store_bytes(int64_t n_seq, int nq_codes) {
  if (n_seq <= 0 || nq_codes <= 0) return 0;
  return (size_t)((n_seq + 1) / 2) * (size_t)((nq_codes + 7) / 8) * 256 * 16;
}

int rqae_search_tc_pack_store(const void* codes, int code_dtype, int64_t code_stride, int64_t n_seq, int seq_len,
                              int nq_codes, int K, void* store_tc, size_t store_bytes, void* stream) {
  if (!codes || !store_tc || n_seq <= 0 || seq_len <= 0 || nq_codes <= 0 || K <= 0 || code_stride < nq_codes) return RQAE_EINVAL;
  if (code_dtype < 0 || code_dtype > 2 || ((uintptr_t)store_tc & 15)) return RQAE_EINVAL;
  if (seq_len > 128 || K + 1 > rq::IT_LUT_ROWS) return RQAE_EUNSUPPORTED;
  if (store_bytes < rqae_search_tc_store_bytes(n_seq, nq_codes)) return RQAE_ESIZE;
  const long long units = (n_seq + 1) / 2;
  if (units >= (1LL << 31)) return RQAE_EUNSUPPORTED;
  const int L8 = (nq_codes + 7) / 8;
  dim3 grid((unsigned)units, (unsigned)(L8 < 8 ? L8 : 8));
  with_code_type(code_dtype, [&](auto tag) {
    using CT = decltype(tag);
    rq::srch_pack_store_kernel<CT><<<grid, 256, 0, (cudaStream_t)stream>>>((const CT*)codes, code_stride, n_seq, seq_len,
                                                                          nq_codes, K, L8, (uint4*)store_tc);
  });
  RQ_CUDA(launched());
  return RQAE_OK;
}

size_t rqae_search_tc_workspace_bytes(const int32_t* layers_host, int n_layers_list) {
  int nkb = 0, last = 0;
  if (srch_tc_nkb(layers_host, n_layers_list, &nkb, &last)) return 0;
  return 4096 + (size_t)nkb * rq::IT_U_TILE;
}

int rqae_search_tc_maxima_f16(const void* store_tc, int64_t n_seq, int seq_len, int nq_codes, const void* vtab_f16,
                              const void* utab_f16, int table_layers, int K, const int32_t* query, int64_t query_stride,
                              int n_query, const int32_t* layers_host, int n_layers_list, void* max_out, int64_t max_stride,
                              void* workspace, size_t workspace_bytes, void* stream) {
  if (!store_tc || !vtab_f16 || !utab_f16 || !query || !max_out || !workspace || n_seq <= 0 || seq_len <= 0 || K <= 0)
    return RQAE_EINVAL;
  if (n_query <= 0 || n_query > rq::IT_FT || seq_len > 128 || K + 1 > rq::IT_LUT_ROWS) return RQAE_EUNSUPPORTED;
  int nkb = 0, last = 0;
  int rc = srch_tc_nkb(layers_host, n_layers_list, &nkb, &last);
  if (rc) return rc;
  const int L8 = (nq_codes + 7) / 8;
  if (last > nq_codes || query_stride < last || table_layers < 8 * ((last + 7) / 8)) return RQAE_EINVAL;   // the tables are padded to whole blocks
  const long long units = (n_seq + 1) / 2;
  if (max_stride < 2 * units || (max_stride & 7) || ((uintptr_t)max_out & 15)) return RQAE_EINVAL;         // the layout the selection reads
  if (((uintptr_t)workspace & 1023) || workspace_bytes < rqae_search_tc_workspace_bytes(layers_host, n_layers_list)) return RQAE_ESIZE;
  if (((uintptr_t)store_tc & 15) || ((uintptr_t)vtab_f16 & 15) || ((uintptr_t)utab_f16 & 15)) return RQAE_EINVAL;
  int sms = 0;
  rc = device_sm_count(&sms);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* ws = (unsigned char*)workspace;
  rq::SrchPrepParams pp;
  memset(&pp, 0, sizeof(pp));
  for (int c = 0; c < n_layers_list; c++) pp.ends[c] = layers_host[c];
  pp.n_cuts = n_layers_list; pp.sched = (rq::IntKBlock*)ws;
  rq::srch_prep_kernel<<<1, 32, 0, st>>>(pp);
  RQ_CUDA(launched());
  {
    const int total = nkb * rq::IT_FT * 8;
    rq::srch_pack_u_kernel<<<(total + 255) / 256, 256, 0, st>>>(query, query_stride, n_query, last, K, (const uint4*)utab_f16,
                                                               (const rq::IntKBlock*)ws, nkb, ws + 4096);
    RQ_CUDA(launched());
  }
  // leave the rest of the SM's 256 KB to L1: the factor gathers re-use sectors within a K-block
  RQ_CUDA(ensure_func_attr((const void*)rq::rq_intensity_kernel<2>, cudaFuncAttributePreferredSharedMemoryCarveout, 58));
  rq::IntParams ip;
  memset(&ip, 0, sizeof(ip));
  ip.u_tiles = ws + 4096; ip.sched = (const rq::IntKBlock*)ws; ip.K = K; ip.NKB = nkb; ip.n_cuts = n_layers_list;
  ip.F = n_query; ip.F_tiles = 1; ip.n_tok_tiles = units; ip.L = last; ip.T_pad = units * rq::IT_TOK;
  ip.s_codes = (const uint4*)store_tc; ip.s_vtab = (const uint4*)vtab_f16; ip.s_max = (__half*)max_out;
  ip.s_stride = max_stride; ip.s_len = seq_len; ip.L8 = L8; ip.stagger = 0;
  return launch_gemm<2>(ip, units, sms, nullptr, st);
}

size_t rqae_search_qrows_bytes(int n_layers, int n_query, int K) {
  if (n_layers <= 0 || n_query <= 0 || K <= 0) return 0;
  return (size_t)n_layers * (size_t)n_query * (size_t)K * sizeof(__half);
}

int rqae_search_build_qrows_f16(const void* sims_f16, int K, const int32_t* query, int64_t query_stride, int n_query,
                                int n_layers, void* qrows, size_t qrows_bytes, void* stream) {
  if (!sims_f16 || !query || !qrows || K <= 0 || n_layers <= 0 || n_query <= 0 || query_stride < n_layers) return RQAE_EINVAL;
  if (n_query > rq::SR_Q || n_layers > 65535) return RQAE_EUNSUPPORTED;
  if (qrows_bytes < rqae_search_qrows_bytes(n_layers, n_query, K)) return RQAE_ESIZE;
  dim3 grid((unsigned)n_query, (unsigned)n_layers);
  rq::search_qrows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const __half*)sims_f16, query, query_stride, n_query, n_layers, K,
                                                                  (__half*)qrows);
  RQ_CUDA(launched());
  return RQAE_OK;
}

int rqae_search_rows_f16(const void* table, int K, const void* codes, int code_dtype, int64_t code_stride, int64_t n_seq,
                         int seq_len, const int32_t* sel, int n_query, int n_sel, const int32_t* layers_host,
                         int first_range, int n_cuts, void* rows_out, void* stream) {
  if (!table || !codes || !sel || !rows_out || !layers_host || K <= 0 || n_seq <= 0 || seq_len <= 0) return RQAE_EINVAL;
  if (code_dtype < 0 || code_dtype > 2 || n_query <= 0 || n_sel < 0 || first_range < 0 || n_cuts <= 0) return RQAE_EINVAL;
  if (n_query > rq::SR_Q || first_range + n_cuts > rq::IT_MAX_CUTS) return RQAE_EUNSUPPORTED;
  rq::SearchRowsParams rp;
  memset(&rp, 0, sizeof(rp));
  int a = 0;
  for (int r = 0; r < first_range + n_cuts; r++) {
    if (layers_host[r] <= a) return RQAE_EINVAL;
    rp.ends[r] = a = layers_host[r];
  }
  if (code_stride < a) return RQAE_EINVAL;
  if (n_sel == 0) return RQAE_OK;
  rp.table = (const __half*)table; rp.codes = codes; rp.code_stride = code_stride; rp.n_seq = n_seq; rp.seq_len = seq_len;
  rp.K = K; rp.n_query = n_query; rp.n_sel = n_sel; rp.n_cuts = n_cuts; rp.first_range = first_range; rp.sel = sel;
  rp.out = (__half*)rows_out;
  if (K > rq::SRW_KMAX || n_seq * (int64_t)seq_len >= 0xFFFFFFFFLL) return RQAE_EUNSUPPORTED;
  const unsigned blocks = (unsigned)(n_query * n_cuts);                      // one block per (cut, query position)
  with_code_type(code_dtype, [&](auto tag) {
    rq::search_rows_kernel<decltype(tag)><<<blocks, rq::SRW_THREADS, 0, (cudaStream_t)stream>>>(rp);
  });
  RQ_CUDA(launched());
  return RQAE_OK;
}

// ---------------------------------------------------------------------------------------------
// tensor-core decode (opt-in; rq_decode.cuh is the bit-exact default)
// ---------------------------------------------------------------------------------------------
static int dec_tc_layout(int nq_codes, int dim, int64_t n_tokens, int passes, GemmLayout* o) {
  if (nq_codes <= 0 || dim <= 0 || n_tokens < 0 || (passes != 1 && passes != 3)) return RQAE_EINVAL;
  const int nkb = passes * ((nq_codes + rq::IT_LPB - 1) / rq::IT_LPB);
  if (nkb > rq::IT_MAX_KB) return RQAE_EUNSUPPORTED;
  *o = gemm_layout(nq_codes, nkb, dim, n_tokens, true);
  return RQAE_OK;
}

size_t rqae_decode_tc_workspace_bytes(int nq_codes, int dim, int64_t n_tokens, int passes) {
  GemmLayout L;
  if (dec_tc_layout(nq_codes, dim, n_tokens, passes, &L)) return 0;
  return L.total;
}

int rqae_decode_tc_f32(const float* w_out, const float* b_out, const float* codebook0, int nq, int nq_codes, int dim,
                       int codebook_dim, int K, const void* codes, int code_dtype, int64_t code_stride,
                       const uint8_t* layer_mask, int64_t n_tokens, float* q_out, int passes, void* workspace,
                       size_t workspace_bytes, void* stream) {
  if (!w_out || !b_out || !codebook0 || !codes || !q_out || !workspace || nq <= 0 || nq_codes <= 0 || nq_codes > nq || K <= 0)
    return RQAE_EINVAL;
  if (code_dtype < 0 || code_dtype > 2 || code_stride < nq_codes) return RQAE_EINVAL;
  if (codebook_dim != 4 || K + 1 > rq::IT_LUT_ROWS) return RQAE_EUNSUPPORTED;
  GemmLayout L;
  int rc = dec_tc_layout(nq_codes, dim, n_tokens, passes, &L);
  if (rc) return rc;
  if (((uintptr_t)workspace & 1023) || workspace_bytes < L.total) return RQAE_ESIZE;
  if (n_tokens == 0) return RQAE_OK;
  int sms = 0;
  rc = device_sm_count(&sms);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* ws = (unsigned char*)workspace;
  rq::DecPrepParams pp;
  pp.L = nq_codes; pp.K = K; pp.passes = passes; pp.codebook0 = codebook0;
  pp.sched = (rq::IntKBlock*)(ws + L.off_sched); pp.wcum = (float*)(ws + L.off_wcum); pp.lut = (uint2*)(ws + L.off_lut);
  rq::dec_prep_kernel<<<4, 256, 0, st>>>(pp);
  RQ_CUDA(launched());
  {
    dim3 grid((unsigned)(L.T_pad / rq::IT_TOK), (unsigned)((nq_codes + 31) / 32)), block(256);
    uint32_t* ct = (uint32_t*)(ws + L.off_codes);
    with_code_type(code_dtype, [&](auto tag) {
      using CT = decltype(tag);
      rq::int_transpose_kernel<CT><<<grid, block, 0, st>>>((const CT*)codes, code_stride, n_tokens, nq_codes, K, true, ct);
    });
    RQ_CUDA(launched());
  }
  {
    const long long total = (long long)L.F_tiles * L.NKB * rq::IT_FT * rq::IT_LPB;
    rq::dec_pack_u_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(w_out, dim, L.F_tiles, L.NKB,
                                                                          (const rq::IntKBlock*)(ws + L.off_sched), layer_mask,
                                                                          ws + L.off_u);
    RQ_CUDA(launched());
    rq::dec_bias_kernel<<<(dim + 127) / 128, 128, 0, st>>>(b_out, nq_codes, dim, layer_mask, (float*)(ws + L.off_bias));
    RQ_CUDA(launched());
  }
  rq::IntParams ip;
  memset(&ip, 0, sizeof(ip));
  ip.codes_p = (const uint32_t*)(ws + L.off_codes); ip.L = nq_codes; ip.T_pad = L.T_pad; ip.u_tiles = ws + L.off_u;
  ip.sched = (const rq::IntKBlock*)(ws + L.off_sched); ip.wcum = (const float*)(ws + L.off_wcum);
  ip.lut = (const uint2*)(ws + L.off_lut); ip.K = K; ip.NKB = L.NKB; ip.n_cuts = 1; ip.F = dim; ip.F_tiles = L.F_tiles;
  ip.n_tok_tiles = L.T_pad / rq::IT_TOK; ip.q_out = q_out; ip.bias = (const float*)(ws + L.off_bias); ip.T = n_tokens; ip.D = dim;
  ip.stagger = 0;
  return launch_gemm<1>(ip, L.units(), sms, nullptr, st);   // the decode epilogue stores with plain instructions
}

}  // extern "C"
