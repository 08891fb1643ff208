// Feature intensities for many features at once, as a tcgen05 GEMM over code tensors (sm_100a).
//
// Replaces RQAEFeature.intensity (rqae/feature.py:102-129, reference harish-kamath/rqae) as it is used by the
// mining loop of scripts/3_make_rqae_features.py:98-114: for feature f with center codes center_f[l] and
// token t with codes code_t[l],
//     intensity[t, f, cut] = fp16( fp16( sum_{l <= cut} w_l * sims[center_f[l], code_t[l]] ) / fp16( sum_{l <= cut} w_l ) )
// where sims = (n n^T).half(), n = F.normalize(codebook[0]) (rqae/model.py:140-142) and w_l = the fp16 layer
// weight (feature.py:97-99).  Because sims is the Gram matrix of the 4-wide rows n_c, the numerator is a dense
// contraction over k = (l, j), j < 4:
//     S[f, t] = sum_k U[f, k] * V[t, k],   U[f, 4l+j] = fp16(w_l * n[center_f[l]][j]),   V[t, 4l+j] = fp16(n[code_t[l]][j])
// which is what this kernel computes on the 5th-generation tensor cores (kind::f16, fp32 accumulators in
// TMEM), evaluated as a running prefix at every cut.  The reference rounds every term to fp16 and sums in
// fp32; here the fp16-rounded factors are multiplied exactly and summed in fp32 by the tensor core, so the
// numerators differ by rounding noise (tests state the tolerance); the roundings AFTER the sum -- prefix to
// fp16, fp32 divide by the fp16 weight prefix, quotient to fp16 -- are the reference's own.
//
// One CTA (640 threads = 5 warpgroups, 1 per SM, persistent) computes units of 256 tokens x 256 features (two feature
// tiles of 128 = two 128x256 fp32 accumulators = all 512 TMEM columns):
//   warp 0      U producer : one lane, bulk-TMA copies of pre-swizzled 128x64 fp16 tiles (16 KB) from L2, one ring
//                            stage per tile
//   warp 1      MMA issuer : tcgen05.mma M=128 (features) x N=256 (tokens) x K=16, 4 per tile and K-block, issued by
//                            one elected lane of a warp-uniform loop; owns the TMEM allocation (warps 2-3 idle)
//   warps 4-11  V builders : the token operand never exists in memory: each thread turns the codes of ONE token
//                            (layer-major int16, coalesced) into a 128-byte K-major row through a 4 x fp16 lookup
//                            table in shared memory (four interleaved copies against bank conflicts), written in the
//                            128-byte swizzle the MMA expects.  (Per-role clock counters: 4 builder warps with two
//                            rows each needed 1.9 k clocks per K-block against 1.4 k for the MMAs; two groups of four
//                            warps building alternate K-blocks into one stage each were slower still, 1.9 k, because
//                            a group cannot build under its own stage's MMAs.)
//   warps 12-19 epilogue   : four warps per accumulator.  At a cut the issuer commits that accumulator and goes on
//                            with the other one; the warps pull the running prefix out of TMEM (tcgen05.ld
//                            32x32b.x32) -- tokens 0..127 of a row with only the reference's FIRST rounding (prefix ->
//                            fp16) as packed registers, tokens 128..255 finished into swizzled staging boxes -- and
//                            release the accumulator as soon as the last load has landed.  The stores (TMA tensor stores
//                            of [32 features][64 tokens] boxes of out[f][cut][t]), the remaining roundings of the kept
//                            half and its trip through the same boxes run while the MMAs of the next K-blocks do.
// setmaxnreg gives the control warpgroup 40 registers, the builders 80 and the epilogue 136 per thread.
// The K axis is cut into K-blocks of 16 layers (64 k = one 128-byte swizzle row); a segment between two cuts
// that is not a multiple of 16 layers is padded with zero slots (schedule built by int_prep_kernel).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>

#include "rq_common.cuh"

namespace rq {

constexpr int IT_TOK = 256;                     // tokens per unit = MMA N
constexpr int IT_FT = 128;                      // features per tile = MMA M
constexpr int IT_LPB = 16;                      // layers per K-block (64 k values, 128 bytes of fp16)
constexpr int IT_VSTAGES = 2;                   // token operand: built locally, latency = the builders' own work
constexpr int IT_USTAGES = 4;                   // feature operand: bulk copies from L2, one 16 KB tile per stage (2 K-blocks ahead)
constexpr int IT_V_BYTES = IT_TOK * 128;        // 32 KB
constexpr int IT_U_TILE = IT_FT * 128;          // 16 KB
constexpr int IT_MAX_CUTS = 64;
constexpr int IT_MAX_KB = 200;                  // nq = 1024 in three passes (decode, f16x3) is 192 K-blocks
constexpr int IT_LUT_ROWS = 640;                // codebook rows + the zero row must fit (5^4 + 1); two tables (decode f16x3: hi, lo)
constexpr int IT_LUT_COPIES = 4;                // intensity kernel: interleaved copies of the one table it uses, copy = lane & 3 --
                                                // entry (row, copy) sits in 8-byte bank pair (4 row + copy) & 15, so the 16 lanes of a
                                                // half-warp collide 4-into-4 instead of 16-into-16 (2.1 against 3.1 wavefronts per load)
constexpr int IT_STG_BOX = 32 * 128;            // staged box of a tensor-map store: 32 feature rows x 64 tokens fp16, 128-byte swizzle
constexpr int IT_STG_WARP = 2 * IT_STG_BOX;     // per epilogue warp: its 32 rows x 128 tokens (half of the unit's 256)
constexpr int IT_THREADS = 640;              // 5 warpgroups: control, builders x 2, epilogue x 2 (setmaxnreg re-splits the register file)
constexpr int IT_EPI_WARPS = 8;
// register pool: ptxas compiles for 640 threads at 96 registers = 61 440; setmaxnreg can only re-split that pool
constexpr int IT_REG_CTRL = 40, IT_REG_BUILD = 80, IT_REG_EPI = 136;
static_assert(128 * IT_REG_CTRL + 256 * IT_REG_BUILD + 256 * IT_REG_EPI <= IT_THREADS * 96, "register pool budget");
constexpr int IT_REG_BUILD_S = 112, IT_REG_EPI_S = 104;   // example search: the builders hold two batches of gathered rows, the epilogue only reduces
static_assert(128 * IT_REG_CTRL + 256 * IT_REG_BUILD_S + 256 * IT_REG_EPI_S <= IT_THREADS * 96, "register pool budget");
constexpr int IT_BUILDERS = 256;             // one token row per builder thread

struct IntKBlock {   // one K-block of the schedule: layers l0 .. l0+n-1 (n <= 16), the rest of the 16 slots zero
  int l0, n, cut, tab;   // cut >= 0: this block ends the segment of that cut (the epilogue emits it);
                         // tab: which of the two lookup tables the token operand is built from (decode: 0 hi, 1 lo)
};

struct IntParams {
  const uint32_t* codes_p;       // [T_pad/256][L][128] tile-major codes: word b of (tile, layer) = code(token b) | code(token b+128) << 16;
                                 // out-of-range and padding codes = K (the zero row)
  int L;                         // layers present in codes_p
  long long T_pad;               // multiple of IT_TOK
  const unsigned char* u_tiles;  // [F_tiles][NKB][16 KB]
  const IntKBlock* sched;        // [NKB]
  const float* wcum;             // [n_cuts] float(fp16(sum_{l<=cut} w_l)), then [n_cuts] its fp32 reciprocal
  const uint2* lut;              // [2][IT_LUT_ROWS] fp16x4 codebook rows (table 0; table 1 only in decode f16x3), row K = 0
  int K, NKB, n_cuts, F, F_tiles;
  __half* out;                   // [F][n_cuts][out_stride]
  long long out_stride;
  long long n_tok_tiles;
  // decode epilogue (EPI = 1): q_out[t][d] = accumulator + bias[d], fp32, rows of `D` floats, t < T
  float* q_out;
  const float* bias;
  long long T;
  int D;
  // example-search maxima (EPI = 2): the "features" are the query positions (one tile of 128), the tokens of a unit
  // are two dataset sequences (128 columns each), the token operand is gathered per layer from a factor table
  const uint4* s_codes;   // [n_units][L8][256] rows of 8 int16 codes (8-layer block-major copy of the code store)
  const uint4* s_vtab;    // [L8 * 8][IT_LUT_ROWS] rows of 8 fp16: the dataset-side factors of the layer's table, row K and layers >= L zero
  __half* s_max;          // [n_cuts][128][s_stride]: max over the positions of every sequence
  long long s_stride;     // >= 2 * n_units, even
  int s_len, L8;          // positions per sequence (<= 128), 8-layer blocks per token
  int stagger;            // clocks between the start groups of CTAs (0: all start together)
};

struct IntSmem {
  static constexpr int VRING = 0;
  static constexpr int URING = IT_VSTAGES * IT_V_BYTES;
  static constexpr int STG = URING + IT_USTAGES * IT_U_TILE;   // 1024-byte aligned: the swizzle pattern of the store boxes
  static constexpr int LUT = STG + IT_EPI_WARPS * IT_STG_WARP;
  static constexpr int SCHED = LUT + IT_LUT_COPIES * IT_LUT_ROWS * 8;   // >= the decode kernel's two tables
  static constexpr int WCUM = SCHED + IT_MAX_KB * 16;
  static constexpr int BARS = WCUM + 2 * IT_MAX_CUTS * 4;
  static constexpr int TMEM_PTR = BARS + (2 * IT_VSTAGES + 2 * IT_USTAGES + 4) * 8;
  static constexpr int TOTAL = TMEM_PTR + 16;
};
// Example search (EPI = 2): no staging boxes and no lookup table, three feature-tile stages -- 119 KB, so that the SM keeps
// ~120 KB of L1 for the factor-row gathers (two rows share a 32-byte sector and 8 layers x 640 rows are 80 KB per K-block).
constexpr int IT_USTAGES_S = 3;
struct IntSmemS {
  static constexpr int VRING = 0;
  static constexpr int URING = IT_VSTAGES * IT_V_BYTES;
  static constexpr int STG = 0, LUT = 0;   // unused
  static constexpr int SCHED = URING + IT_USTAGES_S * IT_U_TILE;
  static constexpr int WCUM = SCHED + IT_MAX_KB * 16;
  static constexpr int BARS = WCUM + 2 * IT_MAX_CUTS * 4;
  static constexpr int TMEM_PTR = BARS + (2 * IT_VSTAGES + 2 * IT_USTAGES + 4) * 8;
  static constexpr int TOTAL = TMEM_PTR + 16;
};
static_assert(IntSmemS::TOTAL <= 131 * 1024, "example search: fits the 132 KB carve-out");
template <int EPI> struct IntSmemOf { using type = IntSmem; };
template <> struct IntSmemOf<2> { using type = IntSmemS; };
static_assert(IntSmem::STG % 1024 == 0, "store boxes must be 1024-byte aligned");
static_assert(IntSmem::TOTAL <= 227 * 1024, "shared memory budget");

// ---- tcgen05 wrappers -------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {   // arrives on `bar` when all MMAs issued so far have completed
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// K-major operand tile in the canonical 128-byte-swizzle layout: rows of 128 bytes, 8-row groups 1024 bytes
// apart (SBO), 16-byte chunk index XORed with (row & 7); descriptor version 1 (sm_100), layout type 2.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor: fp16 x fp16 -> fp32, both operands K-major, M x N
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// The reference's post-sum arithmetic for a pair of values: prefix -> fp16, fp32 divide by the fp16 weight
// prefix, quotient -> fp16 (feature.py:123-127 on CPU tensors).  The divide is a multiply by the fp32
// reciprocal: it can differ from the correctly rounded quotient by one fp32 ulp, which changes the fp16
// result for ~2e-4 of the values by one fp16 ulp -- far inside the tolerance of the sum itself.
__device__ __forceinline__ uint32_t finish2(float a, float b, float inv) {
  const float2 p = __half22float2(__floats2half2_rn(a, b));
  const __half2 h = __floats2half2_rn(p.x * inv, p.y * inv);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// The same arithmetic in two steps, so that the first rounding (the reference's own: prefix -> fp16) can be taken while
// the accumulator is still held and the rest after it has been released.
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t finish_packed(uint32_t ph, float inv) {
  const float2 p = __half22float2(*reinterpret_cast<const __half2*>(&ph));
  const __half2 h = __floats2half2_rn(p.x * inv, p.y * inv);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// ---- TMA tensor store: a [32 rows][64 tokens] fp16 box, shared -> global through a 3-D tensor map of out[f][cut][t]
// (SASS: UTMASTG); tracked by the issuing thread's bulk async-group.  One instruction moves 4 KB; rows beyond the
// tensor's extent (features >= F) are clipped by the hardware.
__device__ __forceinline__ void tma_store_box(const CUtensorMap* tmap, uint32_t src_smem, int tok, int cut, int frow, uint64_t policy) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%1, %2, %3}], [%4], %5;" ::"l"(tmap),
               "r"(tok), "r"(cut), "r"(frow), "r"(src_smem), "l"(policy)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}

// one lane of a converged warp (the same one every time): tcgen05.commit tracks the MMAs of the thread that issues it
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// latency-critical waits (MMA issuer, producers): poll without the suspend hint
__device__ __forceinline__ void mbar_wait_spin(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!ok);
}

// EPI = 0: feature intensities (fp16 out[f][cut][t] with the reference's roundings).
// EPI = 1: tensor-core decode -- "features" are the D output dimensions, U holds W_out, one cut at the last layer,
//          out is q_out[t][d] fp32 (+ the summed out-projection biases); opt-in, not bit-exact (rq_decode.cuh is).
template <int EPI>
__global__ void __launch_bounds__(IT_THREADS, 1) rq_intensity_kernel(const IntParams p, const __grid_constant__ CUtensorMap out_map) {
  extern __shared__ __align__(1024) unsigned char smem[];
  using SM = typename IntSmemOf<EPI>::type;
  constexpr int USTAGES = EPI == 2 ? IT_USTAGES_S : IT_USTAGES;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM::BARS);
  uint64_t* v_full = bars;                      // [VS] 128 builder arrivals
  uint64_t* v_empty = v_full + IT_VSTAGES;      // [VS] MMAs reading the stage have completed (tcgen05.commit)
  uint64_t* u_full = v_empty + IT_VSTAGES;      // [US] bulk copies landed
  uint64_t* u_empty = u_full + IT_USTAGES;      // [US] tcgen05.commit
  uint64_t* acc_full = u_empty + IT_USTAGES;    // [2] segment complete in accumulator a (tcgen05.commit)
  uint64_t* acc_free = acc_full + 2;            // [2] the 4 epilogue warps of accumulator a have read it
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + SM::TMEM_PTR);
  const IntKBlock* sched = reinterpret_cast<const IntKBlock*>(smem + SM::SCHED);
  const float* wcum_s = reinterpret_cast<const float*>(smem + SM::WCUM);

  // ---- one-time setup ----
  for (int i = threadIdx.x; i <= p.K && EPI != 2; i += IT_THREADS) {
    if (EPI == 1) {
      reinterpret_cast<uint2*>(smem + SM::LUT)[i] = p.lut[i];
      reinterpret_cast<uint2*>(smem + SM::LUT)[IT_LUT_ROWS + i] = p.lut[IT_LUT_ROWS + i];
    } else {
      const uint2 r = p.lut[i];
#pragma unroll
      for (int t = 0; t < IT_LUT_COPIES; t++) reinterpret_cast<uint2*>(smem + SM::LUT)[i * IT_LUT_COPIES + t] = r;
    }
  }
  for (int i = threadIdx.x; i < p.NKB * 4; i += IT_THREADS)
    reinterpret_cast<int*>(smem + SM::SCHED)[i] = reinterpret_cast<const int*>(p.sched)[i];
  for (int i = threadIdx.x; i < 2 * p.n_cuts && EPI != 2; i += IT_THREADS)
    reinterpret_cast<float*>(smem + SM::WCUM)[i] = p.wcum[i];
  if (threadIdx.x == 0) {
    for (int s = 0; s < IT_VSTAGES; s++) { mbar_init(&v_full[s], IT_BUILDERS); mbar_init(&v_empty[s], 1); }
    for (int s = 0; s < IT_USTAGES; s++) { mbar_init(&u_full[s], 1); mbar_init(&u_empty[s], 1); }
    for (int a = 0; a < 2; a++) { mbar_init(&acc_full[a], 1); mbar_init(&acc_free[a], IT_EPI_WARPS / 2); }
    mbar_fence_init();
  }
  if (warp == 1) {   // TMEM: all 512 columns (1 CTA per SM)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  const int n_pairs = (p.F_tiles + 1) / 2;
  const long long n_units = p.n_tok_tiles * n_pairs;
  if (p.stagger > 0) {
    // De-phase the CTAs: the first ten cuts of scripts/3's list fall into the first ten K-blocks of a unit, so every
    // unit begins with a burst of output (1.3 MB per SM) and, started together, all SMs burst together and wait on
    // HBM writes.  Four start groups a fraction of a unit apart spread the bursts (measured: 1.73 -> 1.63 ms).
    constexpr int IT_STAGGER_GROUPS = 4;
    const long long t0 = clock64();
    const long long d = (long long)(blockIdx.x % IT_STAGGER_GROUPS) * p.stagger;
    while (clock64() - t0 < d) {
    }
    __syncthreads();
  }
  const uint32_t vring = smem_u32(smem + SM::VRING), uring = smem_u32(smem + SM::URING);
  if (vring & 1023u) __trap();   // the hand-written swizzle assumes 1024-byte aligned tiles

  // (each setmaxnreg sits at the top of its role's branch: ptxas budgets the code it dominates)
  if (warp < 4) {
    reg_dec<IT_REG_CTRL>();
  if (warp == 0) {
    // ======================= U producer =======================
    if (lane == 0) {
      uint32_t s = 0, par = 1;   // a fresh barrier passes a wait on parity 1
      for (long long u = blockIdx.x; u < n_units; u += gridDim.x) {
        const int pr = (int)(u % n_pairs);
        const int nft = min(2, p.F_tiles - 2 * pr);
        for (int kb = 0; kb < p.NKB; kb++) {
          for (int ft = 0; ft < nft; ft++) {
            mbar_wait_spin(&u_empty[s], par);
            mbar_arrive_expect_tx(&u_full[s], IT_U_TILE);
            tma_bulk_g2s(uring + s * IT_U_TILE, p.u_tiles + ((size_t)(2 * pr + ft) * p.NKB + kb) * (size_t)IT_U_TILE, IT_U_TILE,
                         &u_full[s]);
            if (++s == USTAGES) { s = 0; par ^= 1; }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ======================= MMA issuer =======================
    // The whole warp runs the loop (uniform control flow: descriptors, stage counters and barrier addresses stay in
    // uniform registers) and ONE elected lane issues the MMAs and commits.  With the loop under `if (lane == 0)` the
    // compiler moved every operand through ELECT / R2UR sequences: ~290 dependent instructions per K-block, more
    // than the MMAs themselves take (ncu source view, profiles/r2r_intensity_stalls.txt).
    {
      constexpr uint32_t idesc = umma_idesc_f16(IT_FT, IT_TOK);
      uint32_t vs = 0, vpar = 0, us = 0, upar = 0;
      uint32_t free_par0 = 0, free_par1 = 0;
      bool pend0 = false, pend1 = false;   // accumulator a was handed to its epilogue warps and not yet taken back
      for (long long u = blockIdx.x; u < n_units; u += gridDim.x) {
        const int pr = (int)(u % n_pairs);
        const int nft = min(2, p.F_tiles - 2 * pr);
        for (int kb = 0; kb < p.NKB; kb++) {
          const bool is_cut = sched[kb].cut >= 0;
          mbar_wait_spin(&v_full[vs], vpar);
          const uint64_t bd = umma_desc_sw128(vring + vs * IT_V_BYTES);
#pragma unroll
          for (int ft = 0; ft < 2; ft++) {
            if (ft >= nft) break;
            mbar_wait_spin(&u_full[us], upar);
            bool& pend = ft ? pend1 : pend0;
            uint32_t& free_par = ft ? free_par1 : free_par0;
            if (pend) {   // the epilogue of the previous cut (or of the previous unit's last cut) still owns this accumulator
              mbar_wait_spin(&acc_free[ft], free_par);
              free_par ^= 1;
              pend = false;
            }
            tc_fence_after();
            const uint64_t ad = umma_desc_sw128(uring + us * IT_U_TILE);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < 4; k++)   // 16 k values = 32 bytes inside the swizzle row: start address += 2 (x16 B)
                umma_f16(tmem_base + ft * IT_TOK, ad + 2 * k, bd + 2 * k, idesc, (kb | k) != 0);
              tc_commit(&u_empty[us]);
              if (is_cut) tc_commit(&acc_full[ft]);   // the running prefix goes to its epilogue warps; the other accumulator carries on
            }
            __syncwarp();
            if (++us == USTAGES) { us = 0; upar ^= 1; }
            pend = is_cut;
          }
          if (elect_one()) tc_commit(&v_empty[vs]);
          __syncwarp();
          if (++vs == IT_VSTAGES) { vs = 0; vpar ^= 1; }
        }
      }
    }
  }   // warps 2-3: spare warps of the control warpgroup
  } else if (warp < 12) {
    // ======================= V builders =======================
    if constexpr (EPI == 2) reg_inc<IT_REG_BUILD_S>(); else reg_dec<IT_REG_BUILD>();
    if constexpr (EPI == 2) {
      // Example search: row b of the tile is position (b & 127) of sequence 2 u + (b >> 7); a K-block is 8 layers x 8 fp16,
      // one 16-byte factor row per (token, layer) gathered from the L2-resident table.  Per step: store the rows gathered
      // during the previous step, hand the stage over, then request the next step's rows (their codes were loaded a step
      // earlier) and the codes of the step after that.
      const int b = threadIdx.x - 128;
      const uint32_t row_off = b * 128;
      const uint32_t sw = (uint32_t)(b & 7);
      uint32_t s = 0, par = 1;
      struct Pos { long long u; int kb; };
      auto next = [&](Pos& q) { if (++q.kb == p.NKB) { q.kb = 0; q.u += gridDim.x; } };
      auto load_codes = [&](const Pos& q) -> uint4 {
        if (q.u >= n_units) return make_uint4(0u, 0u, 0u, 0u);
        return __ldg(p.s_codes + ((size_t)q.u * p.L8 + sched[q.kb].l0) * IT_TOK + b);
      };
      auto gather = [&](uint4 (&g)[8], const uint4& c, const Pos& q) {
        if (q.u >= n_units) return;
        const uint4* tab = p.s_vtab + (size_t)sched[q.kb].l0 * 8 * IT_LUT_ROWS;
        const uint32_t w[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
        for (int i = 0; i < 8; i++) g[i] = __ldg(tab + (size_t)i * IT_LUT_ROWS + ((w[i >> 1] >> ((i & 1) * 16)) & 0xFFFFu));
      };
      // two batches of gathers in flight: the rows stored in step k were requested in step k - 2
      Pos cur = {(long long)blockIdx.x, 0}, p1 = cur, p2, p3;
      next(p1);
      p2 = p1;
      next(p2);
      p3 = p2;
      next(p3);
      uint4 gA[8], gB[8];
      gather(gA, load_codes(cur), cur);
      gather(gB, load_codes(p1), p1);
      uint4 cn = load_codes(p2);
      auto do_step = [&](uint4 (&g)[8]) {
        mbar_wait_spin(&v_empty[s], par);
        const uint32_t vb = vring + s * IT_V_BYTES + row_off;
#pragma unroll
        for (int i = 0; i < 8; i++)
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(vb + (((uint32_t)i ^ sw) << 4)), "r"(g[i].x), "r"(g[i].y),
                       "r"(g[i].z), "r"(g[i].w)
                       : "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_arrive(&v_full[s]);
        if (++s == IT_VSTAGES) { s = 0; par ^= 1; }
        gather(g, cn, p2);
        cn = load_codes(p3);
        cur = p1;
        p1 = p2;
        p2 = p3;
        next(p3);
      };
      while (cur.u < n_units) {
        do_step(gA);
        if (cur.u >= n_units) break;
        do_step(gB);
      }
    } else {
    const int b = threadIdx.x - 128;   // row b of the token tile
    const uint32_t lut = smem_u32(smem + SM::LUT) + (EPI == 0 ? (uint32_t)(lane & (IT_LUT_COPIES - 1)) * 8u : 0u);
    constexpr uint32_t lut_pitch = EPI == 0 ? 8u * IT_LUT_COPIES : 8u;
    const uint32_t row_off = b * 128;
    const uint32_t sw = (uint32_t)(b & 7);
    const uint32_t csh = (uint32_t)(b >> 7) * 16u;   // the code word holds token (b & 127) in its low and token (b & 127) + 128 in its high half
    uint32_t s = 0, par = 1;
    // The codes of a K-block are 16 coalesced 128-byte warp loads.  They are requested TWO K-blocks ahead into
    // registers, and the K-block IT_PF steps ahead is pulled into L2 with one bulk prefetch: the code rows stream
    // from HBM and their latency must stay off the V hand-over path.
    struct Pos { long long u; int kb; long long tile; };   // tile = u / n_pairs, divided once per unit (a 64-bit division per K-block showed up as ~400 clocks)
    auto next = [&](Pos& q) { if (++q.kb == p.NKB) { q.kb = 0; q.u += gridDim.x; q.tile = q.u / n_pairs; } };
    auto fetch = [&](uint32_t (&c)[IT_LPB], const Pos& q) {
      const uint32_t padw = (uint32_t)p.K | ((uint32_t)p.K << 16);
      if (q.u < n_units) {
        const int l0 = sched[q.kb].l0, n = sched[q.kb].n;
        const uint32_t* src = p.codes_p + ((size_t)q.tile * p.L + l0) * 128 + (b & 127);
#pragma unroll
        for (int i = 0; i < IT_LPB; i++) c[i] = (i < n) ? __ldg(src + i * 128) : padw;
      }
    };
    auto l2_prefetch = [&](const Pos& q) {
      if (b == 0 && q.u < n_units) {
        const int l0 = sched[q.kb].l0, n = sched[q.kb].n;
        const uint32_t* src = p.codes_p + ((size_t)q.tile * p.L + l0) * 128;
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(n * 512) : "memory");
      }
    };
    auto step = [&](uint32_t (&c)[IT_LPB], const Pos& now, Pos& fut, Pos& pf) {
      uint32_t a0[IT_LPB];   // table byte offsets of this block's row
      const uint32_t tsel = (EPI == 1) ? (uint32_t)(sched[now.kb].tab & 1) * (IT_LUT_ROWS * 8u) : 0u;
#pragma unroll
      for (int i = 0; i < IT_LPB; i++) a0[i] = ((c[i] >> csh) & 0xFFFFu) * lut_pitch + tsel;
      fetch(c, fut);
      next(fut);
      l2_prefetch(pf);
      next(pf);
      mbar_wait_spin(&v_empty[s], par);
      const uint32_t vb = vring + s * IT_V_BYTES;
#pragma unroll
      for (int cc = 0; cc < 8; cc++) {
        uint32_t x0, x1, x2, x3;
        asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(x0), "=r"(x1) : "r"(lut + a0[2 * cc]));
        asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(x2), "=r"(x3) : "r"(lut + a0[2 * cc + 1]));
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(vb + row_off + (((uint32_t)cc ^ sw) << 4)), "r"(x0),
                     "r"(x1), "r"(x2), "r"(x3)
                     : "memory");
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the MMA
      mbar_arrive(&v_full[s]);   // (one poller and one arrival per warp instead of all threads was measured: slower, the __syncwarps sit on the hand-over path)
      if (++s == IT_VSTAGES) { s = 0; par ^= 1; }
    };
    constexpr int IT_PF = 8;
    Pos cur = {(long long)blockIdx.x, 0, (long long)blockIdx.x / n_pairs}, fut = cur, pf = cur;
    uint32_t cA[IT_LPB], cB[IT_LPB];
    fetch(cA, fut); next(fut);
    fetch(cB, fut); next(fut);
    for (int i = 0; i < IT_PF; i++) { if (i >= 2) l2_prefetch(pf); next(pf); }
    while (cur.u < n_units) {
      step(cA, cur, fut, pf);
      next(cur);
      if (cur.u >= n_units) break;
      step(cB, cur, fut, pf);
      next(cur);
    }
    }   // EPI != 2
  } else {
    // ======================= epilogue =======================
    reg_inc<(EPI == 2 ? IT_REG_EPI_S : IT_REG_EPI)>();
    const int q = warp & 3;            // TMEM lane quarter this warp may read
    const int acc = (warp - 12) >> 2;   // accumulator (feature tile of the pair)
    uint64_t* const my_full = &acc_full[acc];
    uint64_t* const my_free = &acc_free[acc];
    // The warp's staging area: two store boxes of [32 rows][64 tokens] fp16 (half of the unit's 256 tokens at a time).
    // Lane = feature row; the 16-byte chunk index inside a 128-byte box row is XOR-ed with (row & 7): the 128-byte
    // swizzle the tensor map names, and what keeps the lane-strided 128-bit stores free of bank conflicts.
    const uint32_t wstg = smem_u32(smem + SM::STG) + (uint32_t)(warp - 12) * IT_STG_WARP;
    const uint32_t stg_row = wstg + (uint32_t)lane * 128u;
    const uint32_t stg_x = (uint32_t)(lane & 7);
    auto stg_addr = [&](int j) -> uint32_t {   // chunk j (0..15) of this lane's 128 staged tokens
      return stg_row + (uint32_t)(j >> 3) * IT_STG_BOX + ((((uint32_t)j & 7u) ^ stg_x) << 4);
    };
    const uint64_t pol = l2_policy_evict_first();   // the intensities are a stream: keep the U tiles and code rows in L2
    uint32_t full_par = 0;
    for (long long u = blockIdx.x; u < n_units; u += gridDim.x) {
      const int pr = (int)(u % n_pairs);
      const long long tok0 = (u / n_pairs) * IT_TOK;
      const int nft = min(2, p.F_tiles - 2 * pr);
      if (acc >= nft) continue;   // no such feature tile: the issuer does not signal this accumulator in this unit
      for (int kb = 0; kb < p.NKB; kb++) {
        const int cut = sched[kb].cut;
        if (cut < 0) continue;
        mbar_wait(my_full, full_par);   // idle most of the time: suspended wait, no polling traffic next to the builders
        full_par ^= 1;
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * IT_TOK;
        if (EPI == 2) {
          // example search: lane = query position, columns = the positions of two sequences; out = max over positions
          float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll 2   // fully unrolled, ptxas keeps more TMEM loads in flight than the registers hold and spills
          for (int ch = 0; ch < IT_TOK / 32; ch++) {
            uint32_t v[32];
            tmem_ld32(taddr + ch * 32, v);
            tmem_ld_wait();
            if (ch == IT_TOK / 32 - 1) {
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(my_free);
            }
            float m = -INFINITY;
#pragma unroll
            for (int j = 0; j < 32; j++)
              if (((ch & 3) * 32 + j) < p.s_len) m = fmaxf(m, __uint_as_float(v[j]));
            if (ch < 4) m0 = fmaxf(m0, m); else m1 = fmaxf(m1, m);
          }
          const __half2 r = __floats2half2_rn(m0, m1);
          *reinterpret_cast<__half2*>(p.s_max + ((size_t)cut * IT_FT + q * 32 + lane) * (size_t)p.s_stride + 2 * u) = r;
          continue;
        }
        if (EPI == 1) {
          // decode: lane = output dimension d, columns = tokens; a store instruction covers 32 consecutive floats
          const int d = (2 * pr + acc) * IT_FT + q * 32 + lane;
          const float bsum = d < p.D ? __ldg(p.bias + d) : 0.f;
#pragma unroll 1
          for (int ch = 0; ch < IT_TOK / 32; ch++) {
            uint32_t v[32];
            tmem_ld32(taddr + ch * 32, v);
            tmem_ld_wait();
            if (ch == IT_TOK / 32 - 1) {
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(my_free);
            }
            float* o = p.q_out + (size_t)(tok0 + ch * 32) * p.D + d;
            if (d < p.D) {
#pragma unroll
              for (int j = 0; j < 32; j++)
                if (tok0 + ch * 32 + j < p.T) __stcs(o + (size_t)j * p.D, __uint_as_float(v[j]) + bsum);
            }
          }
          continue;
        }
        const float inv = wcum_s[p.n_cuts + cut];
        const int frow0 = (2 * pr + acc) * IT_FT + q * 32;   // the warp's 32 feature rows; rows >= F are clipped by the tensor map
        const bool do_store = lane == 0;
        // (1) tokens 0..127 of the row: only the reference's FIRST rounding (prefix -> fp16), kept packed in registers;
        // (2) tokens 128..255: finished and staged (the boxes have been read by the previous cut's stores: that wait
        // sits at the bottom of this loop, not inside the hold).
        uint32_t keep[64];
#pragma unroll
        for (int ch = 0; ch < 4; ch++) {
          uint32_t v[32];
          tmem_ld32(taddr + ch * 32, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; j++) keep[ch * 16 + j] = pack_h2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
        }
#pragma unroll 2   // fully unrolled, ptxas keeps more TMEM loads in flight than the registers hold and spills the kept half
        for (int ch = 4; ch < 8; ch++) {
          uint32_t v[32];
          tmem_ld32(taddr + ch * 32, v);
          tmem_ld_wait();
          if (ch == 7) {   // the whole prefix has left TMEM: the issuer may accumulate into it again
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(my_free);
          }
#pragma unroll
          for (int g = 0; g < 4; g++)   // all roundings at once: every trip through shared memory competes with the operand traffic
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg_addr((ch - 4) * 4 + g)),
                         "r"(finish2(__uint_as_float(v[8 * g + 0]), __uint_as_float(v[8 * g + 1]), inv)),
                         "r"(finish2(__uint_as_float(v[8 * g + 2]), __uint_as_float(v[8 * g + 3]), inv)),
                         "r"(finish2(__uint_as_float(v[8 * g + 4]), __uint_as_float(v[8 * g + 5]), inv)),
                         "r"(finish2(__uint_as_float(v[8 * g + 6]), __uint_as_float(v[8 * g + 7]), inv))
                         : "memory");
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the TMA store
        __syncwarp();
        if (do_store) {
          tma_store_box(&out_map, wstg, (int)tok0 + 128, cut, frow0, pol);
          tma_store_box(&out_map, wstg + IT_STG_BOX, (int)tok0 + 192, cut, frow0, pol);
        }
        if (lane == 0) bulk_commit();
        // (4) the kept half: remaining roundings in registers while the first stores drain, then the same boxes again
#pragma unroll
        for (int j = 0; j < 64; j++) keep[j] = finish_packed(keep[j], inv);
        if (lane == 0) bulk_wait_read_all();
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 16; j++)
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg_addr(j)), "r"(keep[4 * j]), "r"(keep[4 * j + 1]),
                       "r"(keep[4 * j + 2]), "r"(keep[4 * j + 3])
                       : "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (do_store) {
          tma_store_box(&out_map, wstg, (int)tok0, cut, frow0, pol);
          tma_store_box(&out_map, wstg + IT_STG_BOX, (int)tok0 + 64, cut, frow0, pol);
        }
        if (lane == 0) bulk_commit();
        // the boxes must have been read before the next cut's prefix is staged: wait here, not while holding TMEM
        if (lane == 0) bulk_wait_read_all();
        __syncwarp();
      }
    }
    if (lane == 0) bulk_wait_all();   // the boxes are read, and the rows written, before the CTA retires
    __syncwarp();
  }

  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------
// preparation kernels (once per call; tiny next to the GEMM)
// ---------------------------------------------------------------------------------------------------
struct IntPrepParams {
  int cuts[IT_MAX_CUTS];
  int n_cuts, K;
  const float* cb_norm;            // [K][4] F.normalize(codebook[0])
  const __half* w;                 // [L] fp16 layer weights
  IntKBlock* sched;
  float* wcum;                     // [2 * n_cuts]
  uint2* lut;                      // [K + 1]
};

// block 0 thread 0: schedule + weight prefixes (sequential fp32 sum, every prefix rounded to fp16, as
// torch's CPU cumsum on a Half tensor does); all threads: the fp16 lookup table.
__global__ void int_prep_kernel(const IntPrepParams p) {
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  for (int c = gid; c <= p.K; c += gridDim.x * blockDim.x) {
    uint2 r = make_uint2(0u, 0u);
    if (c < p.K) {
      const float4 v = reinterpret_cast<const float4*>(p.cb_norm)[c];
      const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
      r = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
    }
    p.lut[c] = r;
  }
  if (gid != 0) return;
  int kb = 0, prev = -1;
  float run = 0.f;
  int l = 0;
  for (int c = 0; c < p.n_cuts; c++) {
    const int cut = p.cuts[c];
    for (int l0 = prev + 1; l0 <= cut; l0 += IT_LPB) {
      const int n = min(IT_LPB, cut - l0 + 1);
      IntKBlock b;
      b.l0 = l0; b.n = n; b.cut = (l0 + n - 1 == cut) ? c : -1; b.tab = 0;
      p.sched[kb++] = b;
    }
    for (; l <= cut; l++) run = __fadd_rn(run, __half2float(p.w[l]));
    const float wc = __half2float(__float2half_rn(run));
    p.wcum[c] = wc;
    p.wcum[p.n_cuts + c] = __fdiv_rn(1.0f, wc);
    prev = cut;
  }
}

// codes [T][stride] (int16 / int32 / int64) -> tile-major int16 pairs [T_pad/256][L][128][2]: within a tile of 256
// tokens the codes of token b and token b+128 at one layer share a 32-bit word (the two rows one builder thread
// writes), and a tile's layers are contiguous (one bulk L2 prefetch per K-block).  Out-of-range codes and the
// padding tokens map to K (the zero row of the lookup table).  wrap_negative (decode): a code in [-K, 0) first takes the
// python-style index c + K, as codebook[0][codes] and the bit-exact decode do.
template <typename CT>
__global__ void __launch_bounds__(256) int_transpose_kernel(const CT* __restrict__ codes, long long stride, long long T, int L,
                                                            int K, bool wrap_negative, uint32_t* __restrict__ out) {
  // block = one token tile (256 tokens) x 32 layers, staged in shared memory as [token][layer] with an 80-byte pitch
  __shared__ __align__(16) unsigned char tile[IT_TOK * 80];
  const long long tt = blockIdx.x;
  const long long t0 = tt * IT_TOK;
  const int l0 = blockIdx.y * 32;
  const int tid = threadIdx.x;
  const bool vec = sizeof(CT) == 2 && (stride % 8) == 0 && ((uintptr_t)codes % 16) == 0 && l0 + 32 <= L;
  if (vec) {   // int16 codes: 16-byte loads (8 layers of one token), four per thread
#pragma unroll
    for (int it = 0; it < 4; it++) {
      const int idx = tid + it * 256;
      const int i = idx >> 2, c = idx & 3;   // token, 16-byte chunk of its 32 layers
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      const bool live = t0 + i < T;
      if (live) v = __ldg(reinterpret_cast<const uint4*>(codes + (t0 + i) * stride + l0) + c);
      uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; k++) {
        int lo = (short)(w[k] & 0xFFFFu), hi = (short)(w[k] >> 16);
        if (wrap_negative) { lo += lo < 0 ? K : 0; hi += hi < 0 ? K : 0; }
        lo = (!live || lo < 0 || lo >= K) ? K : lo;
        hi = (!live || hi < 0 || hi >= K) ? K : hi;
        w[k] = (uint32_t)lo | ((uint32_t)hi << 16);
      }
      *reinterpret_cast<uint4*>(tile + i * 80 + c * 16) = make_uint4(w[0], w[1], w[2], w[3]);
    }
  } else {
    for (int idx = tid; idx < IT_TOK * 32; idx += 256) {
      const int i = idx >> 5, j = idx & 31;
      unsigned short v = (unsigned short)K;
      if (t0 + i < T && l0 + j < L) {
        long long c = (long long)codes[(t0 + i) * stride + l0 + j];
        if (wrap_negative && c < 0) c += K;
        if (c >= 0 && c < K) v = (unsigned short)c;
      }
      *reinterpret_cast<unsigned short*>(tile + i * 80 + j * 2) = v;
    }
  }
  __syncthreads();
  // word b of (tile, layer) = code(token b) | code(token b + 128) << 16: a warp writes 128 contiguous bytes
  for (int idx = tid; idx < 32 * 128; idx += 256) {
    const int j = idx >> 7, b = idx & 127;
    if (l0 + j >= L) continue;
    const uint32_t lo = *reinterpret_cast<const unsigned short*>(tile + b * 80 + j * 2);
    const uint32_t hi = *reinterpret_cast<const unsigned short*>(tile + (b + 128) * 80 + j * 2);
    out[((size_t)tt * L + l0 + j) * 128 + b] = lo | (hi << 16);
  }
}

// U tiles: [F_tiles][NKB] tiles of 128 features x 64 k fp16 in the swizzled K-major layout;
// U[f][4 s + j] = fp16(float(w_l) * n[center_f[l]][j]) for slot s < n of the K-block (l = l0 + s), else 0
__global__ void int_pack_u_kernel(const int* __restrict__ centers, long long center_stride, int F, int F_tiles, int NKB,
                                  const IntKBlock* __restrict__ sched, const float* __restrict__ cb_norm, int K,
                                  const __half* __restrict__ w, unsigned char* __restrict__ u_tiles) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)F_tiles * NKB * IT_FT * IT_LPB;
  if (gid >= total) return;
  const int s = (int)(gid % IT_LPB);
  const int r = (int)((gid / IT_LPB) % IT_FT);
  const int kb = (int)((gid / (IT_LPB * IT_FT)) % NKB);
  const int ft = (int)(gid / ((long long)IT_LPB * IT_FT * NKB));
  const IntKBlock b = sched[kb];
  const int f = ft * IT_FT + r;
  uint2 val = make_uint2(0u, 0u);
  if (f < F && s < b.n) {
    const int l = b.l0 + s;
    const int c = centers[(size_t)f * center_stride + l];
    if (c >= 0 && c < K) {
      const float wl = __half2float(w[l]);
      const float4 v = reinterpret_cast<const float4*>(cb_norm)[c];
      const __half2 a = __floats2half2_rn(wl * v.x, wl * v.y), bb = __floats2half2_rn(wl * v.z, wl * v.w);
      val = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&bb));
    }
  }
  unsigned char* tile = u_tiles + ((size_t)ft * NKB + kb) * (size_t)IT_U_TILE;
  const int chunk = s >> 1;
  *reinterpret_cast<uint2*>(tile + r * 128 + (((chunk ^ (r & 7)) << 4) | ((s & 1) << 3))) = val;
}

// ---------------------------------------------------------------------------------------------------
// tensor-core decode (EPI = 1): preparation kernels
// ---------------------------------------------------------------------------------------------------
// q[t][d] = sum_l sum_j c[t][l][j] * W_out[l][d][j] + sum_l b_out[l][d]  (rqae/model.py:232-252) as the same GEMM:
// V[t][4l+j] = codebook[0][code_t[l]][j], U[d][4l+j] = W_out[l][d][j].  One pass rounds both factors to fp16
// (relative error of q ~2e-4); three passes add the fp16 remainders: V_hi U_hi + V_hi U_lo + V_lo U_hi (~2e-5: what is
// left is the tensor core's fp32 accumulation over 3 x 4096 terms).
// K-block tab: bit 0 = token operand from the remainder table, bit 1 = weight operand is the remainder.
struct DecPrepParams {
  int L, K, passes;
  const float* codebook0;   // [K][4]
  IntKBlock* sched;
  float* wcum;
  uint2* lut;               // [2][IT_LUT_ROWS]
};

__device__ __forceinline__ uint2 pack_h4(float a, float b, float c, float d) {
  const __half2 x = __floats2half2_rn(a, b), y = __floats2half2_rn(c, d);
  return make_uint2(*reinterpret_cast<const uint32_t*>(&x), *reinterpret_cast<const uint32_t*>(&y));
}
__device__ __forceinline__ float h_rem(float v) { return v - __half2float(__float2half_rn(v)); }

__global__ void dec_prep_kernel(const DecPrepParams p) {
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  for (int c = gid; c <= p.K; c += gridDim.x * blockDim.x) {
    uint2 hi = make_uint2(0u, 0u), lo = hi;
    if (c < p.K) {
      const float4 v = reinterpret_cast<const float4*>(p.codebook0)[c];
      hi = pack_h4(v.x, v.y, v.z, v.w);
      lo = pack_h4(h_rem(v.x), h_rem(v.y), h_rem(v.z), h_rem(v.w));
    }
    p.lut[c] = hi;
    p.lut[IT_LUT_ROWS + c] = lo;
  }
  if (gid != 0) return;
  int kb = 0;
  for (int ps = 0; ps < p.passes; ps++) {
    for (int l0 = 0; l0 < p.L; l0 += IT_LPB) {
      IntKBlock b;
      b.l0 = l0; b.n = min(IT_LPB, p.L - l0); b.cut = -1; b.tab = ps == 0 ? 0 : (ps == 1 ? 2 : 1);
      p.sched[kb++] = b;
    }
  }
  p.sched[kb - 1].cut = 0;
  p.wcum[0] = 1.0f;
  p.wcum[1] = 1.0f;
}

// weight operand tiles: [F_tiles][NKB] tiles of 128 output dimensions x 64 k, same swizzled layout as the feature tiles
__global__ void dec_pack_u_kernel(const float* __restrict__ w_out, int D, int F_tiles, int NKB,
                                  const IntKBlock* __restrict__ sched, const unsigned char* __restrict__ layer_mask,
                                  unsigned char* __restrict__ u_tiles) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)F_tiles * NKB * IT_FT * IT_LPB;
  if (gid >= total) return;
  const int s = (int)(gid % IT_LPB);
  const int r = (int)((gid / IT_LPB) % IT_FT);
  const int kb = (int)((gid / (IT_LPB * IT_FT)) % NKB);
  const int ft = (int)(gid / ((long long)IT_LPB * IT_FT * NKB));
  const IntKBlock b = sched[kb];
  const int d = ft * IT_FT + r;
  uint2 val = make_uint2(0u, 0u);
  if (d < D && s < b.n) {
    const int l = b.l0 + s;
    if (layer_mask == nullptr || layer_mask[l]) {
      const float4 w = reinterpret_cast<const float4*>(w_out)[(size_t)l * D + d];
      val = (b.tab & 2) ? pack_h4(h_rem(w.x), h_rem(w.y), h_rem(w.z), h_rem(w.w)) : pack_h4(w.x, w.y, w.z, w.w);
    }
  }
  unsigned char* tile = u_tiles + ((size_t)ft * NKB + kb) * (size_t)IT_U_TILE;
  const int chunk = s >> 1;
  *reinterpret_cast<uint2*>(tile + r * 128 + (((chunk ^ (r & 7)) << 4) | ((s & 1) << 3))) = val;
}

// bias[d] = sum over the selected layers of b_out[l][d], in layer order
__global__ void dec_bias_kernel(const float* __restrict__ b_out, int L, int D, const unsigned char* __restrict__ layer_mask,
                                float* __restrict__ bias) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  float acc = 0.f;
  for (int l = 0; l < L; l++)
    if (layer_mask == nullptr || layer_mask[l]) acc = __fadd_rn(acc, b_out[(size_t)l * D + d]);
  bias[d] = acc;
}

}  // namespace rq
