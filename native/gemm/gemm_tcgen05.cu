// tcgen05 / TMEM / TMA GEMM for sm_100a (hand-written PTX, no CUTLASS dependency).
//
//   C[M,N] (bf16) = A[M,K] (bf16, K contiguous) x B[N,K]^T (bf16, K contiguous)  (+ bias[N])
//   optional fused epilogue: per-column sum / sum-of-squares of the bf16-rounded output
//   accumulated into stats[2*N] (fp32) — the train-mode BatchNorm statistics of a 1x1
//   convolution come for free with the GEMM instead of costing another pass over C.
//
// Structure (one persistent CTA per SM, 256 threads, warp-specialised):
//   warp 0   TMA producer : cp.async.bulk.tensor 2D loads of 128xBK (A) and BNxBK (B) tiles, 128B swizzle,
//                           STAGES-deep mbarrier ring
//   warp 1   MMA issuer   : one elected thread issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=BN, K=16)
//                           from shared-memory descriptors into a TMEM accumulator; tcgen05.commit frees
//                           the smem stage / publishes the accumulator
//   warp 2   TMEM allocator (2 x BN columns = two accumulator stages, so the epilogue of tile i overlaps
//                           the main loop of tile i+1)
//   warps 4-7 epilogue    : tcgen05.ld (32 lanes x 32 columns per warp-instruction) -> bias -> bf16 ->
//                           128B-swizzled staging tile in smem -> TMA store; column statistics are read back
//                           from the staging tile (conflict-free) and kept in registers across the CTA's
//                           tiles of one N-block, flushed with 4 atomics per thread.
// Out-of-bounds rows/columns are handled by TMA (zero fill on load, clipping on store).
//
// K10 (SURVEY.md §2E): the `peer` epilogue mode adds the tile into every rank's output over NVLink
// (multimem.red through the switch = GEMM + all-reduce in one kernel) — see gemm_epilogue.cuh notes below.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <atomic>
#include <type_traits>
#include "device_sync.cuh"   // cross-GPU block barrier shared with libshipyard_coll

namespace {

constexpr int BM = 128;          // UMMA M (cta_group::1)
constexpr int BK = 64;           // one 128-byte swizzle row of bf16
constexpr int UK = 16;           // UMMA K for 16-bit inputs
constexpr int kThreads = 256;
constexpr int kEpiGroups = 2;                             // TN / conv kernel: two epilogue warpgroups drain alternate 64-column chunks
constexpr int kThreadsTN = 128 + kEpiGroups * 128;        // warps 0-3: TMA / MMA / TMEM alloc / idle, then 4 warps per epilogue group
constexpr int kEpiThreads = 128;
constexpr int kEpiChunk = 64;    // columns per epilogue step (one 128B row of bf16)

#ifndef DEVI
#define DEVI __device__ __forceinline__
#endif

DEVI uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ---------------------------------------------------------------------------------
DEVI void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
DEVI void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
DEVI void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded wait: a protocol bug must end in a trap (an error the host sees), never in a box that hangs until it is killed.
DEVI void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t a = smem_u32(bar);
  uint32_t ok, it = 0;
  unsigned long long t0 = 0;
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(a), "r"(parity) : "memory");
    if (!ok && ((++it) & 0x3fff) == 0) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      if (t0 == 0) t0 = t;
      else if (t - t0 > 4000000000ull) {
        asm volatile("trap;");        // surfaces as a launch failure on the host (no device printf: it costs stack + spills)
      }
    }
  } while (!ok);
}
DEVI void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
DEVI void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- TMA ---------------------------------------------------------------------------------------
DEVI void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)tmap) : "memory");
}
DEVI void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(smem_u32(smem_dst)), "l"((uint64_t)tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
// im2col-mode load (4D NHWC activation): `pixels` consecutive base pixels starting at (w, h, n), walking W then H then N
// inside the descriptor's bounding box, `channels` wide from channel c; (off_w, off_h) is the filter tap added to every
// base pixel; taps that land in the padding are zero-filled by the TMA unit.  Lands as [pixels rows x 128 B], 128B swizzle —
// byte-identical to a 2D tile load of a K-major operand, so the convolution needs no materialised im2col matrix.
DEVI void tma_load_im2col_4d(void* smem_dst, const void* tmap, uint64_t* bar, int c, int w, int h, int n, uint16_t off_w, uint16_t off_h) {
  asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};"
               ::"r"(smem_u32(smem_dst)), "l"((uint64_t)tmap), "r"(smem_u32(bar)), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h) : "memory");
}
DEVI void tma_load_3d(void* smem_dst, const void* tmap, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(smem_u32(smem_dst)), "l"((uint64_t)tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
DEVI void tma_store_2d(const void* tmap, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"((uint64_t)tmap), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1) : "memory");
}
DEVI void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> DEVI void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
DEVI void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

DEVI void st_global_v4(void* p, const uint4& v) {
  asm volatile("st.global.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ---- tcgen05 ------------------------------------------------------------------------------------
template <int NCOLS> DEVI void tmem_alloc(uint32_t* dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(NCOLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS> DEVI void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
DEVI void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
DEVI void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
DEVI void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
               ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
DEVI void umma_commit(uint64_t* bar) {   // arrives on `bar` once every MMA issued so far has completed
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
DEVI void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {   // 32 lanes x 32 consecutive fp32 columns
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
               "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
               "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                 "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
                 "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
                 "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
               : "r"(taddr) : "memory");
}
DEVI void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// shared-memory matrix descriptor: K-major operand, 128-byte swizzle, rows of 128 B, 8-row groups 1024 B apart
DEVI uint64_t make_kmajor_sw128_desc(const void* smem_tile) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_u32(smem_tile) & 0x3FFFF) >> 4);   // start address      bits [0,14)
  d |= (uint64_t)1 << 16;                                  // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                        // stride byte offset  bits [32,46)
  d |= (uint64_t)1 << 46;                                  // descriptor version 1 (Blackwell)
  d |= (uint64_t)2 << 61;                                  // layout type: SWIZZLE_128B
  return d;
}
// MN-major operand (the M/N index is the contiguous one), 128-byte swizzle.  Canonical layout in 16-byte units
// ((8,n),(8,k)):((1,LBO),(8,SBO)): a 64-element MN slab is one 128 B row per k; 8 k-rows form a 1024 B swizzle
// group (SBO); the next 64-element MN slab starts LBO bytes later.  Each slab is exactly what one TMA box
// {64 elements, BK rows} with SWIZZLE_128B writes.
DEVI uint64_t make_mnmajor_sw128_desc(const void* smem_tile, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_u32(smem_tile) & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
constexpr int kSlabBytes = 64 * BK * 2;   // one MN-major slab: 64 MN elements x BK k-rows = 8 KB
// instruction descriptor: D=f32, A=B=bf16, M=128, N=BN; bit 15 / 16 = A / B is MN-major
template <int BN, bool kAMN = false, bool kBMN = false> DEVI constexpr uint32_t make_idesc() {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((kAMN ? 1u : 0u) << 15) | ((kBMN ? 1u : 0u) << 16) |
         ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

DEVI void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
DEVI uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
DEVI bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// Implicit-GEMM convolution geometry (kConv): GEMM row m = output pixel (n, p, q), GEMM k = (tap, channel block).
struct ConvGeom {
  int P, Q;          // output height / width
  int S, taps;       // filter width, R*S
  int cblocks;       // A-operand channels / 64
  int stride, lower; // base pixel of output (p, q) = (lower + stride*p, lower + stride*q)
  int flip;          // dgrad: B is W[co][taps-1-tap][ci] read through a 3D map as an MN-major operand
};

// Tile rasterisation: tiles are numbered in groups of kGroupM row-blocks x all column-blocks, row-block fastest inside a group.
// The ~148 tiles in flight at any time then touch only ~kGroupM row-blocks of A and ~148/kGroupM column-blocks of B, which
// fit in the 126 MB L2 — with the plain row-fastest order a large A (or the activations of a wide 1x1 conv) is streamed from
// HBM once per column-block.
constexpr int kGroupM = 16;
DEVI void tile_to_mn(int t, int num_m, int num_n, int& m_blk, int& n_blk) {
  const int per_group = kGroupM * num_n;
  const int g = t / per_group, r = t - g * per_group;
  const int first_m = g * kGroupM;
  const int gm = (num_m - first_m) < kGroupM ? (num_m - first_m) : kGroupM;
  m_blk = first_m + r % gm;
  n_blk = r / gm;
}

// Kernels that accumulate per-column statistics want every CTA to stay on ONE column-block (the partial sums live in registers
// and are flushed with atomics when the column-block changes): tiles are numbered column-block fastest and the persistent
// stride is rounded down to a multiple of num_n, so CTA c always works on column-block c % num_n while the CTAs running
// concurrently still share their A row-blocks through L2.
template <bool kColumnSticky> DEVI void map_tile(int t, int num_m, int num_n, int& m_blk, int& n_blk) {
  if constexpr (kColumnSticky) { m_blk = t / num_n; n_blk = t - m_blk * num_n; }
  else tile_to_mn(t, num_m, num_n, m_blk, n_blk);
}
template <bool kColumnSticky> DEVI void tile_walk(int cta, int ncta, int num_n, int num_tiles, int& t_first, int& t_stride) {
  t_stride = ncta; t_first = cta;
  if constexpr (kColumnSticky) {
    if (ncta >= num_n) { t_stride = ncta - ncta % num_n; if (cta >= t_stride) t_first = num_tiles; }
  }
}

template <int BN> struct Cfg {
  static constexpr int kABytes = BM * BK * 2;                 // 16 KB
  static constexpr int kBBytes = BN * BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kCBytes = BM * kEpiChunk * 2;          // 16 KB staging tile (x2 buffers)
  static constexpr int kBudget = 227 * 1024 - 1024 - 256 - 512;   // opt-in max dynamic smem minus alignment slack and barriers
  static constexpr int kStages = ((kBudget - 2 * kCBytes) / kStageBytes) > 6 ? 6 : ((kBudget - 2 * kCBytes) / kStageBytes);
  static constexpr int kTmemCols = 2 * BN < 32 ? 32 : 2 * BN; // two accumulator stages (power of two: BN in {64,128,256})
  static constexpr int kSmemBytes = kStages * kStageBytes + 2 * kCBytes + 1024 /*align slack*/ + 256 /*barriers*/;
};

// kDirect: the output tile leaves through coalesced 16-byte st.global from the staging buffer instead of a TMA store.  Reason
// (profiles/conv_halo.md, "epilogue"): on the short-K GEMMs of ResNet (K = 64..512, one to eight k-blocks per tile) every 128x64
// epilogue chunk costs 1.7-2 us although TMEM -> registers -> smem is ~0.3 us of work: the group's single staging buffer may
// only be rewritten once the previous TMA store has READ it (`cp.async.bulk.wait_group.read 0`), and that store queues in the
// SM's TMA unit behind the producer's loads for the next 4-6 stages.  Plain stores have no such dependency.
// [round 2, gpurun_out/r2_bench_direct.json: as a global switch the step gets slower (21.10 vs 20.81 ms), so it is selected only with
// SHIPYARD_GEMM_DIRECT_STORE=1 and by the 1x1 / stride-2 dgrad, whose scattering epilogue needs plain stores]
// kEpiAlt (BN = 64, with kDirect): a 64-column tile has one epilogue chunk, so warpgroup g drains accumulator stage g (alternate
// tiles) instead of group 1 idling — same schedule as conv3x3_halo_kernel's kEpiAlt.  [numerics verified on hardware in round 2; selected with
// SHIPYARD_GEMM_DIRECT_STORE=1 SHIPYARD_GEMM_EPI_ALT=1]
// Folded-BatchNorm epilogue (kAffine, inference): out[m, n] = act(acc[m, n] * scale[n] + shift[n] (+ residual[m, n])), all in fp32 on
// the accumulator and rounded to bf16 once.  The residual (bf16, the output's NHWC layout, row pitch ldr) is read by the thread that owns
// the output row, 16 bytes per load, before it waits for the accumulator.  Runs with the st.global store phase (kDirect).
struct EpiAffine {
  const float* scale;                 // [N] fp32, 16-byte aligned
  const float* shift;                 // [N] fp32, 16-byte aligned
  const __nv_bfloat16* residual;      // [M, ldr] or null; never the output itself
  int ldr;
  int relu;
};

template <int BN, bool kStats, bool kBias, bool kBMN = false, bool kConv = false, bool kDirect = false, bool kEpiAlt = false,
          bool kAffine = false>
__global__ void __launch_bounds__(kThreadsTN, 1)
gemm_bf16_tn_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                    const __grid_constant__ CUtensorMap tmap_c, int M, int N, int K,
                    const __nv_bfloat16* __restrict__ bias, float* __restrict__ stats, const ConvGeom geom,
                    __nv_bfloat16* __restrict__ c_ptr = nullptr, int ldc = 0, const EpiAffine aff = EpiAffine{}) {
  static_assert(!kAffine || (kDirect && !kStats && !kBias && !kBMN && !kEpiAlt), "kAffine: plain forward GEMM / conv with the st.global epilogue");
  using C = Cfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + C::kStages * C::kABytes;
  uint8_t* smem_c = smem + C::kStages * C::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_c + 2 * C::kCBytes);
  uint64_t* full_bar = bars;                        // [kStages]  TMA -> MMA
  uint64_t* empty_bar = bars + C::kStages;          // [kStages]  MMA -> TMA
  uint64_t* tmem_full = bars + 2 * C::kStages;      // [2]        MMA -> epilogue
  uint64_t* tmem_empty = bars + 2 * C::kStages + 2; // [2]        epilogue -> MMA
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * C::kStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_m = (M + BM - 1) / BM, num_n = (N + BN - 1) / BN, num_k = (K + BK - 1) / BK;
  const int num_tiles = num_m * num_n;
  int t_first, t_stride;
  tile_walk<kStats>(blockIdx.x, gridDim.x, num_n, num_tiles, t_first, t_stride);

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmap_a); tma_prefetch_desc(&tmap_b); tma_prefetch_desc(&tmap_c); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    constexpr int kActiveGroups = (BN / kEpiChunk) < kEpiGroups ? (BN / kEpiChunk) : kEpiGroups;
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], kEpiThreads * kActiveGroups); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<C::kTmemCols>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int t = t_first; t < num_tiles; t += t_stride) {
        int m_blk, n_blk; map_tile<kStats>(t, num_m, num_n, m_blk, n_blk);
        int cn = 0, ch = 0, cw = 0;
        if constexpr (kConv) {               // first output pixel of this M tile -> base-pixel coordinates
          const int pq = geom.P * geom.Q, m0 = m_blk * BM;
          cn = m0 / pq; const int rem = m0 - cn * pq, p0 = rem / geom.Q;
          ch = geom.lower + geom.stride * p0; cw = geom.lower + geom.stride * (rem - p0 * geom.Q);
        }
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          int nb = BN / 64;
          if constexpr (kBMN) { nb = 0; for (int sl = 0; sl < BN / 64; ++sl) nb += (n_blk * BN + sl * 64 < N); }
          mbar_expect_tx(&full_bar[stage], kBMN ? (uint32_t)(C::kABytes + nb * kSlabBytes) : (uint32_t)C::kStageBytes);
          if constexpr (kConv) {
            const int tap = kb / geom.cblocks, cb = kb - tap * geom.cblocks, r = tap / geom.S, sx = tap - r * geom.S;
            tma_load_im2col_4d(smem_a + stage * C::kABytes, &tmap_a, &full_bar[stage], cb * 64, cw, ch, cn, (uint16_t)sx, (uint16_t)r);
            if constexpr (kBMN) {           // dgrad: B[k = co, n = ci] = W[co][taps-1-tap][ci], 3D map {ci, tap, co}
              for (int sl = 0; sl < nb; ++sl)
                tma_load_3d(smem_b + stage * C::kBBytes + sl * kSlabBytes, &tmap_b, &full_bar[stage], n_blk * BN + sl * 64,
                            geom.flip ? geom.taps - 1 - tap : tap, cb * 64);
            } else {
              tma_load_2d(smem_b + stage * C::kBBytes, &tmap_b, &full_bar[stage], kb * BK, n_blk * BN);
            }
            if (++stage == C::kStages) { stage = 0; phase ^= 1; }
            continue;
          }
          tma_load_2d(smem_a + stage * C::kABytes, &tmap_a, &full_bar[stage], kb * BK, m_blk * BM);
          if constexpr (kBMN) {
            // B given as [K, N] with N contiguous (e.g. W[Cout, Cin] for dgrad): one 64-wide slab per TMA box;
            // slabs entirely past N are skipped (they only feed output columns the TMA store clips)
            for (int sl = 0; sl < nb; ++sl)
              tma_load_2d(smem_b + stage * C::kBBytes + sl * kSlabBytes, &tmap_b, &full_bar[stage], n_blk * BN + sl * 64, kb * BK);
          } else {
            tma_load_2d(smem_b + stage * C::kBBytes, &tmap_b, &full_bar[stage], kb * BK, n_blk * BN);
          }
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc<BN, false, kBMN>();
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int t = t_first; t < num_tiles; t += t_stride) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);       // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&full_bar[stage], phase);             // TMA bytes have landed
          tc_fence_after();
          const uint64_t adesc = make_kmajor_sw128_desc(smem_a + stage * C::kABytes);
          const uint64_t bdesc = kBMN ? make_mnmajor_sw128_desc(smem_b + stage * C::kBBytes, kSlabBytes)
                                      : make_kmajor_sw128_desc(smem_b + stage * C::kBBytes);
          // K advance: K-major = +32 bytes inside the 128B swizzle atom; MN-major = +16 k-rows x 128 B
          constexpr uint64_t kBStep = kBMN ? (UK * 128 >> 4) : (UK * 2 >> 4);
#pragma unroll
          for (int k = 0; k < BK / UK; ++k) {
            umma_bf16(d_tmem, adesc + (uint64_t)(k * UK * 2 >> 4), bdesc + (uint64_t)k * kBStep, idesc, (kb | k) != 0);
          }
          umma_commit(&empty_bar[stage]);                 // smem stage reusable once these MMAs retire
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[acc]);                     // accumulator complete -> epilogue
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue: two warpgroups, TMEM lane quarter = warp % 4 =====================
    // Group g drains chunks g, g+2, ... of every tile through its own staging buffer, so the TMEM-read latency,
    // the smem round trip and the TMA store of one chunk overlap with the other group's chunk; inside a group the
    // tcgen05.ld of the next chunk is issued as soon as the current one has been packed into registers.
    constexpr int kChunks = BN / kEpiChunk;
    static_assert(!kEpiAlt || (BN == kEpiChunk && kDirect), "kEpiAlt: single-chunk tiles with the st.global epilogue");
    const int grp = (warp - 4) >> 2;
    if (grp < kChunks || kEpiAlt) {
      const int cg = kEpiAlt ? 0 : grp;                               // chunk group (kEpiAlt: both groups drain chunk 0 of alternate tiles)
      const int ew = warp & 3, et = threadIdx.x - 128 - grp * 128;   // 0..127 inside the group
      const int row = ew * 32 + lane;                               // row of the 128-row tile owned by this thread
      const bool issuer = et == 0;
      const int bar_a = 1 + 2 * grp, bar_b = 2 + 2 * grp;
      uint8_t* cbuf = smem_c + grp * C::kCBytes;
      int acc = 0; uint32_t acc_phase = 0;
      // statistics: thread (wcol = et % 32, rgrp = et / 32) owns word-column wcol (2 bf16 columns) of rows rgrp*32..+31
      constexpr int kMyChunks = (kChunks + kEpiGroups - 1) / kEpiGroups;
      float st[kMyChunks][4];
#pragma unroll
      for (int c = 0; c < kMyChunks; ++c) { st[c][0] = st[c][1] = st[c][2] = st[c][3] = 0.f; }
      int cur_n = -1;
      auto flush_stats = [&](int n_blk) {
        if (!kStats || n_blk < 0) return;
        const int wcol = et & 31;
#pragma unroll
        for (int ci = 0; ci < kMyChunks; ++ci) {
          const int c = cg + ci * kEpiGroups;
          if (c < kChunks) {
            const int col = n_blk * BN + c * kEpiChunk + 2 * wcol;
            if (col < N) { atomicAdd(&stats[col], st[ci][0]); atomicAdd(&stats[N + col], st[ci][2]); }
            if (col + 1 < N) { atomicAdd(&stats[col + 1], st[ci][1]); atomicAdd(&stats[N + col + 1], st[ci][3]); }
          }
          st[ci][0] = st[ci][1] = st[ci][2] = st[ci][3] = 0.f;
        }
      };
      for (int t = t_first; t < num_tiles; t += t_stride) {
        if constexpr (kEpiAlt) {                           // accumulator stage `acc` belongs to warpgroup `acc`
          if (acc != grp) { if (++acc == 2) { acc = 0; acc_phase ^= 1; } continue; }
        }
        int m_blk, n_blk; map_tile<kStats>(t, num_m, num_n, m_blk, n_blk);
        if (kStats && n_blk != cur_n) { flush_stats(cur_n); cur_n = n_blk; }
        mbar_wait(&tmem_full[acc], acc_phase);
        tc_fence_after();
        const uint32_t tbase = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * BN);
        uint32_t v[2][32];
        tmem_ld32(tbase + cg * kEpiChunk, v[0]);
        tmem_ld32(tbase + cg * kEpiChunk + 32, v[1]);
#pragma unroll
        for (int ci = 0; ci < kMyChunks; ++ci) {
          const int c = cg + ci * kEpiGroups;
          if (c >= kChunks) break;
          uint4 rsd[8];                     // kAffine: this row's 64 residual columns, loaded while the TMEM read is in flight
          if constexpr (kAffine) {
            const int mrow = m_blk * BM + row, c0 = n_blk * BN + c * kEpiChunk;
#pragma unroll
            for (int q = 0; q < 8; ++q)
              rsd[q] = (aff.residual && mrow < M && c0 + q * 8 < N)
                           ? __ldg(reinterpret_cast<const uint4*>(aff.residual + (size_t)mrow * (size_t)aff.ldr + c0 + q * 8))
                           : make_uint4(0u, 0u, 0u, 0u);
          }
          tmem_ld_wait();
          const bool last = c + kEpiGroups >= kChunks;
          if (last) {                       // this group's part of the accumulator is in registers: hand it back early
            tc_fence_before();
            mbar_arrive(&tmem_empty[acc]);
          }
          const int n0 = n_blk * BN + c * kEpiChunk;
          uint4 w[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {     // 8 x 16-byte chunks = 64 bf16 columns of this thread's row
            float f[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(v[(q * 8 + i) >> 5][(q * 8 + i) & 31]);
            if (kBias) {
#pragma unroll
              for (int i = 0; i < 8; ++i) { const int col = n0 + q * 8 + i; f[i] += col < N ? __bfloat162float(bias[col]) : 0.f; }
            }
            if constexpr (kAffine) {        // N % 8 == 0: a 16-byte piece is wholly inside or wholly past the last column
              if (n0 + q * 8 < N) {
                const float4 s0 = __ldg(reinterpret_cast<const float4*>(aff.scale + n0 + q * 8));
                const float4 s1 = __ldg(reinterpret_cast<const float4*>(aff.scale + n0 + q * 8 + 4));
                const float4 t0 = __ldg(reinterpret_cast<const float4*>(aff.shift + n0 + q * 8));
                const float4 t1 = __ldg(reinterpret_cast<const float4*>(aff.shift + n0 + q * 8 + 4));
                const float s[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
                const float t[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
                const uint32_t rw[4] = {rsd[q].x, rsd[q].y, rsd[q].z, rsd[q].w};
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  const float r = (i & 1) ? __uint_as_float(rw[i >> 1] & 0xffff0000u) : __uint_as_float(rw[i >> 1] << 16);
                  f[i] = fmaf(f[i], s[i], t[i]) + r;
                  if (aff.relu) f[i] = fmaxf(f[i], 0.f);
                }
              }
            }
            w[q] =make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
          }
          if (!last) {                      // prefetch this group's next chunk; its latency hides behind the store phase below
            tmem_ld32(tbase + (c + kEpiGroups) * kEpiChunk, v[0]);
            tmem_ld32(tbase + (c + kEpiGroups) * kEpiChunk + 32, v[1]);
          }
          if constexpr (!kDirect) { if (issuer) tma_store_wait_read<0>(); }   // the previous TMA store of this group has finished reading cbuf
          named_bar_sync(bar_a, kEpiThreads);
#pragma unroll
          for (int q = 0; q < 8; ++q)       // 128B swizzle: 16-byte chunk index XOR (row % 8) — matches the TMA store, bank-conflict free
            *reinterpret_cast<uint4*>(cbuf + row * 128 + ((q ^ (row & 7)) << 4)) = w[q];
          if constexpr (!kDirect) fence_proxy_async_smem();
          named_bar_sync(bar_b, kEpiThreads);
          if constexpr (kDirect) {          // thread (rr = et / 8, sub = et % 8): 16-byte piece `sub` of rows rr, rr + 16, ...: full 128 B lines per 8 lanes
            const int sub = et & 7, rr = et >> 3;
            if (n0 + sub * 8 < N) {
              if (!kConv && geom.stride == 2) {
                // data gradient of a 1x1 / stride-2 convolution: GEMM row (n, p, q) lands on pixel (2p, 2q) of dX[N, 2P, 2Q, ldc] and the
                // three pixels the forward pass skipped get their zeros from the same thread: dX is written exactly once, no memset
                const int pq = geom.P * geom.Q, W2 = 2 * geom.Q;
                const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
                for (int p = 0; p < 8; ++p) {
                  const int r = p * 16 + rr, mrow = m_blk * BM + r;
                  if (mrow < M) {
                    const int img = mrow / pq, rem = mrow - img * pq, py = rem / geom.Q, qx = rem - py * geom.Q;
                    __nv_bfloat16* o = c_ptr + ((size_t)(img * 2 * geom.P + 2 * py) * W2 + 2 * qx) * (size_t)ldc + n0 + sub * 8;
                    st_global_v4(o, *reinterpret_cast<const uint4*>(cbuf + r * 128 + ((sub ^ (r & 7)) << 4)));
                    st_global_v4(o + ldc, z4);
                    st_global_v4(o + (size_t)W2 * ldc, z4);
                    st_global_v4(o + (size_t)(W2 + 1) * ldc, z4);
                  }
                }
              } else {
#pragma unroll
              for (int p = 0; p < 8; ++p) {
                const int r = p * 16 + rr;
                if (m_blk * BM + r < M)
                  st_global_v4(c_ptr + (size_t)(m_blk * BM + r) * (size_t)ldc + n0 + sub * 8,
                               *reinterpret_cast<const uint4*>(cbuf + r * 128 + ((sub ^ (r & 7)) << 4)));
              }
              }
            }
          } else {
            if (issuer) { tma_store_2d(&tmap_c, cbuf, n0, m_blk * BM); tma_store_commit(); }
          }
          if (kStats) {
            const int wcol = et & 31, rgrp = et >> 5;
            const int q = wcol >> 2, wi = wcol & 3;
            const int rows_valid = M - m_blk * BM;          // OOB rows hold zeros from the zero-filled A tile (no bias with stats)
            float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll 8
            for (int r = rgrp * 32; r < rgrp * 32 + 32; ++r) {
              const uint32_t wv = *reinterpret_cast<const uint32_t*>(cbuf + r * 128 + ((q ^ (r & 7)) << 4) + wi * 4);
              const float a = __uint_as_float(wv << 16), b = __uint_as_float(wv & 0xffff0000u);
              if (r < rows_valid) { s0 += a; s1 += b; q0 = fmaf(a, a, q0); q1 = fmaf(b, b, q1); }
            }
            st[ci][0] += s0; st[ci][1] += s1; st[ci][2] += q0; st[ci][3] += q1;
          }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      flush_stats(cur_n);
      if constexpr (!kDirect) { if (issuer) tma_store_wait_all(); }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc<C::kTmemCols>(tmem_base); }
}


// ===================================================================================================
// Weight-gradient GEMM: D[i, j] = sum_k A[k, i] * B[k, j], both operands MN-major (a 1x1-conv / Linear wgrad:
// A = X[pixels, Cin], B = dY[pixels, Cout], D = dW[Cout, Cin] stored as out[j * ldo + i]).  The reduction
// dimension is the huge one (pixels) and the output is tiny, so the work is split along K over all SMs:
// every CTA accumulates its K-range in TMEM, adds the fp32 tile into a workspace with red.global.add, and the
// LAST CTA to finish a tile (atomic ticket) converts it to bf16 straight into the gradient buffer and leaves
// workspace + ticket zeroed for the next launch — one kernel, no split-K reduce pass, no transposes, no
// separate gradient-accumulate kernel, CUDA-graph capturable (no host-side memset).
// ===================================================================================================
DEVI void red_add_f32(float* p, float v) { asm volatile("red.relaxed.gpu.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory"); }

// kConv: A is the im2col view of an NHWC activation with the GEMM's I index = tap * Cin + ci (exactly the KRSC row of dW), so
// each 64-wide A slab is one TMA im2col box of one filter tap: a 128-row tile covers two taps of a 64-channel layer (no wasted
// MMA rows, dY is re-read 5x instead of 9x) and the output needs no per-tap offsets.
template <int BN, bool kConv = false>
__global__ void __launch_bounds__(kThreads, 1)
gemm_bf16_nt_splitk_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                           int I, int J, int K, int splits, float* __restrict__ ws_base, int* __restrict__ tickets,
                           __nv_bfloat16* __restrict__ out_base, int ldo, int accumulate, const ConvGeom geom) {
  using C = Cfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + C::kStages * C::kABytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::kStages * C::kStageBytes + 2 * C::kCBytes);
  uint64_t* full_bar = bars; uint64_t* empty_bar = bars + C::kStages;
  uint64_t* tmem_full = bars + 2 * C::kStages; uint64_t* tmem_empty = bars + 2 * C::kStages + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * C::kStages + 4);
  uint32_t* s_last = tmem_ptr + 1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_m = (I + BM - 1) / BM, num_n = (J + BN - 1) / BN, num_k = (K + BK - 1) / BK;
  const int num_mn = num_m * num_n;
  const int num_items = num_mn * splits;
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmap_a); tma_prefetch_desc(&tmap_b); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], kEpiThreads); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<C::kTmemCols>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int w = blockIdx.x; w < num_items; w += gridDim.x) {
        // K-split-major order: concurrently running CTAs work on the SAME pixel range (K-split) for different output tiles, so
        // x / dY stream from HBM once and are shared through L2 instead of being re-streamed once per tile
        const int tile = w % num_mn, sp = w / num_mn;
        const int n_blk = tile / num_m, m_blk = tile % num_m;
        const int kb0 = (int)((long)sp * num_k / splits), kb1 = (int)((long)(sp + 1) * num_k / splits);
        // slabs that start beyond the matrix edge are not loaded at all: their smem stays stale, which only
        // feeds accumulator rows / columns the epilogue never stores (rows and columns are independent)
        int na = 0, nb = 0;
        for (int sl = 0; sl < BM / 64; ++sl) na += (m_blk * BM + sl * 64 < I);
        for (int sl = 0; sl < BN / 64; ++sl) nb += (n_blk * BN + sl * 64 < J);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_expect_tx(&full_bar[stage], (uint32_t)(na + nb) * kSlabBytes);
          if constexpr (kConv) {           // 64 output pixels starting at linear index kb*64 -> im2col box [64 pixels x 64 channels]
            const int pq = geom.P * geom.Q, m0 = kb * BK;
            const int cn = m0 / pq, rem = m0 - cn * pq, p0 = rem / geom.Q;
            const int ch = geom.lower + geom.stride * p0, cw = geom.lower + geom.stride * (rem - p0 * geom.Q);
            const int cin = geom.cblocks * 64;
            for (int sl = 0; sl < na; ++sl) {
              const int i0 = m_blk * BM + sl * 64, tap = i0 / cin, c0 = i0 - tap * cin, tr = tap / geom.S, ts = tap - tr * geom.S;
              tma_load_im2col_4d(smem_a + stage * C::kABytes + sl * kSlabBytes, &tmap_a, &full_bar[stage], c0, cw, ch, cn,
                                 (uint16_t)ts, (uint16_t)tr);
            }
          } else
          for (int sl = 0; sl < na; ++sl)
            tma_load_2d(smem_a + stage * C::kABytes + sl * kSlabBytes, &tmap_a, &full_bar[stage], m_blk * BM + sl * 64, kb * BK);
          for (int sl = 0; sl < nb; ++sl)
            tma_load_2d(smem_b + stage * C::kBBytes + sl * kSlabBytes, &tmap_b, &full_bar[stage], n_blk * BN + sl * 64, kb * BK);
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc<BN, true, true>();
      int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
      for (int w = blockIdx.x; w < num_items; w += gridDim.x) {
        const int sp = w / num_mn;
        const int kb0 = (int)((long)sp * num_k / splits), kb1 = (int)((long)(sp + 1) * num_k / splits);
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t adesc = make_mnmajor_sw128_desc(smem_a + stage * C::kABytes, kSlabBytes);
          const uint64_t bdesc = make_mnmajor_sw128_desc(smem_b + stage * C::kBBytes, kSlabBytes);
#pragma unroll
          for (int k = 0; k < BK / UK; ++k)       // 16 k-rows x 128 B per UMMA_K step
            umma_bf16(d_tmem, adesc + (uint64_t)(k * UK * 128 >> 4), bdesc + (uint64_t)(k * UK * 128 >> 4), idesc, (kb != kb0) || k != 0);
          umma_commit(&empty_bar[stage]);
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    const int ew = warp - 4, et = threadIdx.x - 128;
    int acc = 0; uint32_t acc_phase = 0;
    for (int w = blockIdx.x; w < num_items; w += gridDim.x) {
      const int tile = w % num_mn;
      const int n_blk = tile / num_m, m_blk = tile % num_m;
      __nv_bfloat16* const out = out_base;
      float* const ws = ws_base;
      const int i = m_blk * BM + ew * 32 + lane;           // TMEM lane = output row i = contiguous index of `out`
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * BN + c * 32), v);
        tmem_ld_wait();
        if (c == BN / 32 - 1) { tc_fence_before(); mbar_arrive(&tmem_empty[acc]); }
        const int j0 = n_blk * BN + c * 32;
        if (i < I) {
          if (splits == 1) {              // whole K in this CTA: write the gradient directly (a warp covers 64 contiguous bytes)
#pragma unroll
            for (int jb = 0; jb < 32; jb += 8) {      // read-modify-write loads in batches of 8: 4 memory round trips, not 32
              float prev[8];
#pragma unroll
              for (int jj = 0; jj < 8; ++jj)
                prev[jj] = (accumulate && j0 + jb + jj < J) ? __bfloat162float(out[(size_t)(j0 + jb + jj) * ldo + i]) : 0.f;
#pragma unroll
              for (int jj = 0; jj < 8; ++jj)
                if (j0 + jb + jj < J) out[(size_t)(j0 + jb + jj) * ldo + i] = __float2bfloat16_rn(__uint_as_float(v[jb + jj]) + prev[jj]);
            }
          } else {
#pragma unroll
            for (int jj = 0; jj < 32; ++jj)
              if (j0 + jj < J) red_add_f32(ws + (size_t)(j0 + jj) * I + i, __uint_as_float(v[jj]));   // one 128 B line per warp instruction
          }
        }
      }
      if (splits > 1) {
        __threadfence();
        named_bar_sync(1, kEpiThreads);
        if (et == 0) *s_last = (atomicAdd(&tickets[tile], 1) == splits - 1) ? 1u : 0u;
        named_bar_sync(2, kEpiThreads);
        if (*s_last) {                                      // every K-split of this tile has been added: finalise it
          __threadfence();
          // thread -> 4 consecutive i (16 B of fp32) x every 4th column; kFin loads in flight per thread so the
          // L2 round trips overlap instead of serialising (I % 8 == 0, so a 4-wide group is all-in or all-out)
          constexpr int kFin = 4;
          const int ii = m_blk * BM + (et & 31) * 4, jsub = et >> 5;
          if (ii < I) {
            for (int jb = 0; jb < BN / 4; jb += kFin) {
              float4 acc4[kFin]; uint2 prev[kFin];
#pragma unroll
              for (int u = 0; u < kFin; ++u) {
                const int j = n_blk * BN + jsub + 4 * (jb + u);
                if (j < J) {
                  acc4[u] = __ldcg(reinterpret_cast<const float4*>(ws + (size_t)j * I + ii));
                  if (accumulate) prev[u] = *reinterpret_cast<const uint2*>(out + (size_t)j * ldo + ii);
                }
              }
#pragma unroll
              for (int u = 0; u < kFin; ++u) {
                const int j = n_blk * BN + jsub + 4 * (jb + u);
                if (j < J) {
                  float4 a = acc4[u];
                  if (accumulate) {
                    a.x += __uint_as_float(prev[u].x << 16); a.y += __uint_as_float(prev[u].x & 0xffff0000u);
                    a.z += __uint_as_float(prev[u].y << 16); a.w += __uint_as_float(prev[u].y & 0xffff0000u);
                  }
                  __stcg(reinterpret_cast<float4*>(ws + (size_t)j * I + ii), make_float4(0.f, 0.f, 0.f, 0.f));
                  *reinterpret_cast<uint2*>(out + (size_t)j * ldo + ii) = make_uint2(pack_bf16(a.x, a.y), pack_bf16(a.z, a.w));
                }
              }
            }
          }
          if (et == 0) tickets[tile] = 0;
        }
        named_bar_sync(1, kEpiThreads);                     // s_last is rewritten by the next item
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc<C::kTmemCols>(tmem_base); }
}

// ===================================================================================================
// K10: GEMM + all-reduce in ONE kernel.  Every rank multiplies its K-shard (C_r = A_r x B_r^T); the
// epilogue adds each fp32 tile straight into the multicast mapping of the output with multimem.red, so the
// NVSwitch applies the addition in every GPU's copy while the next tile's MMAs are already running —
// there is no partial-C round trip through HBM and no separate collective launch.  A cross-GPU flag barrier
// at the end of the kernel makes all contributions visible before any rank's kernel completes.
// `out` must be zero before the first contribution (caller zeroes it and synchronises the ranks).
// ===================================================================================================
DEVI void mc_red_add_v4_f32(void* mc, float a, float b, float c, float d) {
  asm volatile("multimem.red.relaxed.sys.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
DEVI void p2p_red_add_f32(float* p, float v) { asm volatile("red.relaxed.sys.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory"); }

template <int BN>
__global__ void __launch_bounds__(kThreads, 1)
gemm_bf16_tn_allreduce_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                              const __grid_constant__ CommDev comm, size_t out_off, int ldc, int M, int N, int K) {
  using C = Cfg<BN>;
  constexpr int kRowPitch = 32 * 4 + 16;          // 32 fp32 columns + 16 B pad: conflict-free 16 B accesses
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + C::kStages * C::kABytes;
  uint8_t* smem_c = smem + C::kStages * C::kStageBytes;      // 32 KB staging (BM * kRowPitch = 18 KB used)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_c + 2 * C::kCBytes);
  uint64_t* full_bar = bars; uint64_t* empty_bar = bars + C::kStages;
  uint64_t* tmem_full = bars + 2 * C::kStages; uint64_t* tmem_empty = bars + 2 * C::kStages + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * C::kStages + 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_m = (M + BM - 1) / BM, num_n = (N + BN - 1) / BN, num_k = (K + BK - 1) / BK;
  const int num_tiles = num_m * num_n;
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmap_a); tma_prefetch_desc(&tmap_b); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], kEpiThreads); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<C::kTmemCols>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        const int n_blk = t / num_m, m_blk = t % num_m;
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_expect_tx(&full_bar[stage], C::kStageBytes);
          tma_load_2d(smem_a + stage * C::kABytes, &tmap_a, &full_bar[stage], kb * BK, m_blk * BM);
          tma_load_2d(smem_b + stage * C::kBBytes, &tmap_b, &full_bar[stage], kb * BK, n_blk * BN);
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc<BN>();
      int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t adesc = make_kmajor_sw128_desc(smem_a + stage * C::kABytes);
          const uint64_t bdesc = make_kmajor_sw128_desc(smem_b + stage * C::kBBytes);
#pragma unroll
          for (int k = 0; k < BK / UK; ++k)
            umma_bf16(d_tmem, adesc + (uint64_t)(k * UK * 2 >> 4), bdesc + (uint64_t)(k * UK * 2 >> 4), idesc, (kb | k) != 0);
          umma_commit(&empty_bar[stage]);
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    const int ew = warp - 4, et = threadIdx.x - 128;
    const int row = ew * 32 + lane;
    int acc = 0; uint32_t acc_phase = 0;
    char* out_mc = comm.mc ? comm.mc + out_off : nullptr;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      const int n_blk = t / num_m, m_blk = t % num_m;
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      constexpr int kChunks32 = BN / 32;
#pragma unroll 1
      for (int c = 0; c < kChunks32; ++c) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * BN + c * 32), v);
        tmem_ld_wait();
        if (c == kChunks32 - 1) { tc_fence_before(); mbar_arrive(&tmem_empty[acc]); }
        named_bar_sync(1, kEpiThreads);                        // previous chunk fully drained from the staging tile
#pragma unroll
        for (int q = 0; q < 8; ++q)
          *reinterpret_cast<uint4*>(smem_c + row * kRowPitch + q * 16) = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        named_bar_sync(2, kEpiThreads);
        const int n0 = n_blk * BN + c * 32;
#pragma unroll
        for (int i = 0; i < 8; ++i) {                          // coalesced: 8 consecutive threads cover one 128 B row segment
          const int idx = i * kEpiThreads + et, r = idx >> 3, q = idx & 7;
          const int grow = m_blk * BM + r, gcol = n0 + q * 4;
          if (grow < M && gcol < N) {
            const float4 f = *reinterpret_cast<const float4*>(smem_c + r * kRowPitch + q * 16);
            const size_t eoff = ((size_t)grow * ldc + gcol) * sizeof(float);
            if (out_mc) mc_red_add_v4_f32(out_mc + eoff, f.x, f.y, f.z, f.w);     // one op, reduced in every GPU's copy by the switch
            else {
              for (int p = 0; p < comm.world; ++p) {
                float* dst = reinterpret_cast<float*>(comm.heap[p] + out_off + eoff);
                p2p_red_add_f32(dst, f.x); p2p_red_add_f32(dst + 1, f.y); p2p_red_add_f32(dst + 2, f.z); p2p_red_add_f32(dst + 3, f.w);
              }
            }
          }
        }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    __threadfence_system();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc<C::kTmemCols>(tmem_base); }
  // every rank's contributions are in flight or landed: publish + wait for all peers (one flag per CTA)
  uint32_t ep = epoch_load(comm);
  block_barrier(comm, ep);
  epoch_store(comm, ep);
}

// ===================================================================================================
// K10 v2: GEMM + all-reduce with a reduce-scatter / all-gather schedule and bf16 on the wire.
// The multimem.red version above makes every GPU receive N full-size fp32 contributions (ingress = N x |C|),
// which is NVLink-bound at 8 GPUs.  Here every output row-block has an OWNER rank:
//   phase 1  mainloop + epilogue: each rank's partial tile goes (bf16, plain 128 B P2P stores straight from the
//            TMEM read-back, overlapped with the next tile's MMAs) into inbox[src] on the tile's owner
//            -> ingress per GPU = (N-1)/N x |C| x 2 B
//   barrier  cross-GPU flag barrier per CTA + a local grid barrier (all CTAs of all ranks have published)
//   phase 2  the owner sums its N inbox slices in fp32 and multicasts the bf16 result to every GPU with
//            multimem.st (P2P stores when NVLS is unavailable) -> ingress per GPU = (N-1)/N x |C| x 2 B
//   barrier  so nobody's kernel completes before its copy of C is complete.
// One launch, no partial C in the local HBM, fp32 accumulation of the cross-rank sum.
// ===================================================================================================
__device__ unsigned g_gb_count = 0;
__device__ unsigned g_gb_gen = 0;

DEVI void grid_barrier(const CommDev& c) {          // all CTAs are co-resident (persistent grid <= #SMs, 1 CTA/SM)
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned gen;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(gen) : "l"(&g_gb_gen) : "memory");
    __threadfence();
    if (atomicAdd(&g_gb_count, 1u) == gridDim.x - 1) {
      g_gb_count = 0;
      __threadfence();
      asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(&g_gb_gen) : "memory");
    } else {
      unsigned cur, it = 0; unsigned long long t0 = 0;
      do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(cur) : "l"(&g_gb_gen) : "memory");
        if (((++it) & 0x3ff) == 0) {
          const unsigned long long t = globaltimer_ns();
          if (t0 == 0) t0 = t;
          else if (t - t0 > c.timeout_ns) { *reinterpret_cast<volatile uint32_t*>(c.status) = SY_ERR_TIMEOUT; __threadfence_system(); break; }
        }
      } while (cur == gen);
    }
  }
  __syncthreads();
}
DEVI void mc_st_v4(void* mc, const uint4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

struct InboxMaps { CUtensorMap m[SY_MAXR]; };     // one 2-D map per owner rank over ITS inbox (peer-mapped virtual addresses)

template <int BN>
__global__ void __launch_bounds__(kThreadsTN, 1)
gemm_bf16_tn_rsag_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                         const __grid_constant__ InboxMaps inbox_maps, const __grid_constant__ CommDev comm, size_t inbox_off,
                         size_t out_off, int M, int N, int K, int rows_per_rank) {
  using C = Cfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + C::kStages * C::kABytes;
  uint8_t* smem_c = smem + C::kStages * C::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_c + 2 * C::kCBytes);
  uint64_t* full_bar = bars; uint64_t* empty_bar = bars + C::kStages;
  uint64_t* tmem_full = bars + 2 * C::kStages; uint64_t* tmem_empty = bars + 2 * C::kStages + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * C::kStages + 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_m = (M + BM - 1) / BM, num_n = (N + BN - 1) / BN, num_k = (K + BK - 1) / BK;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a); tma_prefetch_desc(&tmap_b);
    for (int p = 0; p < comm.world; ++p) tma_prefetch_desc(&inbox_maps.m[p]);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    constexpr int kActiveGroups = (BN / kEpiChunk) < kEpiGroups ? (BN / kEpiChunk) : kEpiGroups;
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], kEpiThreads * kActiveGroups); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<C::kTmemCols>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  // tile order: owners interleaved (tile t -> owner t % world first), so at any moment the CTAs of one rank push to
  // all peers at once instead of all hammering the same owner's NVLink port
  const int m_per_rank = rows_per_rank / BM;
  auto tile_coords = [&](int t, int& m_blk, int& n_blk) {
    const int per_owner = m_per_rank * num_n;                 // tiles per owner (owners past the matrix edge own fewer)
    const int o = t % comm.world, q = t / comm.world;
    // rotate by my rank so rank r starts on owner r+1 (spreads the first wave)
    const int owner = (o + comm.rank + 1) % comm.world;
    m_blk = owner * m_per_rank + q / num_n; n_blk = q % num_n;
    (void)per_owner;
  };
  const int virt_tiles = m_per_rank * num_n * comm.world;     // includes tiles past M (skipped)

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int t = blockIdx.x; t < virt_tiles; t += gridDim.x) {
        int m_blk, n_blk; tile_coords(t, m_blk, n_blk);
        if (m_blk >= num_m) continue;
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_expect_tx(&full_bar[stage], C::kStageBytes);
          tma_load_2d(smem_a + stage * C::kABytes, &tmap_a, &full_bar[stage], kb * BK, m_blk * BM);
          tma_load_2d(smem_b + stage * C::kBBytes, &tmap_b, &full_bar[stage], kb * BK, n_blk * BN);
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc<BN>();
      int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
      for (int t = blockIdx.x; t < virt_tiles; t += gridDim.x) {
        int m_blk, n_blk; tile_coords(t, m_blk, n_blk);
        if (m_blk >= num_m) continue;
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t adesc = make_kmajor_sw128_desc(smem_a + stage * C::kABytes);
          const uint64_t bdesc = make_kmajor_sw128_desc(smem_b + stage * C::kBBytes);
#pragma unroll
          for (int k = 0; k < BK / UK; ++k)
            umma_bf16(d_tmem, adesc + (uint64_t)(k * UK * 2 >> 4), bdesc + (uint64_t)(k * UK * 2 >> 4), idesc, (kb | k) != 0);
          umma_commit(&empty_bar[stage]);
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // epilogue: two warpgroups drain alternate 64-column chunks; each chunk goes TMEM -> bf16 -> swizzled staging tile -> ONE
    // bulk TMA store into the owner's inbox (peer memory over NVLink, or local HBM for tiles this rank owns)
    constexpr int kChunks = BN / kEpiChunk;
    const int grp = (warp - 4) >> 2;
    if (grp < kChunks) {
      const int ew = warp & 3, et = threadIdx.x - 128 - grp * 128;
      const int row = ew * 32 + lane;
      const bool issuer = et == 0;
      const int bar_a = 1 + 2 * grp, bar_b = 2 + 2 * grp;
      uint8_t* cbuf = smem_c + grp * C::kCBytes;
      constexpr int kMyChunks = (kChunks + kEpiGroups - 1) / kEpiGroups;
      int acc = 0; uint32_t acc_phase = 0;
      for (int t = blockIdx.x; t < virt_tiles; t += gridDim.x) {
        int m_blk, n_blk; tile_coords(t, m_blk, n_blk);
        if (m_blk >= num_m) continue;
        const int owner = m_blk / m_per_rank;
        const int inbox_row0 = comm.rank * rows_per_rank + (m_blk * BM - owner * rows_per_rank);   // [src rank][local row] on the owner
        mbar_wait(&tmem_full[acc], acc_phase);
        tc_fence_after();
        const uint32_t tbase = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * BN);
        uint32_t v[2][32];
        tmem_ld32(tbase + grp * kEpiChunk, v[0]);
        tmem_ld32(tbase + grp * kEpiChunk + 32, v[1]);
#pragma unroll
        for (int ci = 0; ci < kMyChunks; ++ci) {
          const int c = grp + ci * kEpiGroups;
          if (c >= kChunks) break;
          tmem_ld_wait();
          const bool last = c + kEpiGroups >= kChunks;
          if (last) { tc_fence_before(); mbar_arrive(&tmem_empty[acc]); }
          uint4 w[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float f[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(v[(q * 8 + i) >> 5][(q * 8 + i) & 31]);
            w[q] = make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
          }
          if (!last) {
            tmem_ld32(tbase + (c + kEpiGroups) * kEpiChunk, v[0]);
            tmem_ld32(tbase + (c + kEpiGroups) * kEpiChunk + 32, v[1]);
          }
          if (issuer) tma_store_wait_read<0>();
          named_bar_sync(bar_a, kEpiThreads);
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<uint4*>(cbuf + row * 128 + ((q ^ (row & 7)) << 4)) = w[q];
          fence_proxy_async_smem();
          named_bar_sync(bar_b, kEpiThreads);
          if (issuer) { tma_store_2d(&inbox_maps.m[owner], cbuf, n_blk * BN + c * kEpiChunk, inbox_row0); tma_store_commit(); }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      if (issuer) tma_store_wait_all();         // every bulk store of this group has been performed (not just read from smem)
      __threadfence_system();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc<C::kTmemCols>(tmem_base); }

  uint32_t ep = epoch_load(comm);
  block_barrier(comm, ep);          // CTA b of every rank has published its partial tiles
  grid_barrier(comm);               // ... and so have all my sibling CTAs => every contribution to my rows is in my inbox

  // ---- phase 2: reduce my rows over the N inbox slices (fp32) and multicast the bf16 result ----
  const int my_row0 = comm.rank * rows_per_rank;
  int my_rows = M - my_row0; if (my_rows > rows_per_rank) my_rows = rows_per_rank; if (my_rows < 0) my_rows = 0;
  const int vec_per_row = N / 8;
  const long total = (long)my_rows * vec_per_row;
  const __nv_bfloat16* inbox = reinterpret_cast<const __nv_bfloat16*>(comm.heap[comm.rank] + inbox_off);
  for (long idx = (long)blockIdx.x * kThreadsTN + threadIdx.x; idx < total; idx += (long)gridDim.x * kThreadsTN) {
    const int r = (int)(idx / vec_per_row), c8 = (int)(idx % vec_per_row);
    float acc8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    uint4 in[SY_MAXR];
#pragma unroll
    for (int src = 0; src < SY_MAXR; ++src)
      if (src < comm.world) in[src] = __ldcg(reinterpret_cast<const uint4*>(inbox + ((size_t)src * rows_per_rank + r) * N + c8 * 8));
#pragma unroll
    for (int src = 0; src < SY_MAXR; ++src) {
      if (src < comm.world) {
        const uint32_t w[4] = {in[src].x, in[src].y, in[src].z, in[src].w};
#pragma unroll
        for (int i = 0; i < 4; ++i) { acc8[2 * i] += __uint_as_float(w[i] << 16); acc8[2 * i + 1] += __uint_as_float(w[i] & 0xffff0000u); }
      }
    }
    const uint4 o = make_uint4(pack_bf16(acc8[0], acc8[1]), pack_bf16(acc8[2], acc8[3]), pack_bf16(acc8[4], acc8[5]), pack_bf16(acc8[6], acc8[7]));
    const size_t eoff = out_off + ((size_t)(my_row0 + r) * N + c8 * 8) * 2;
    if (comm.mc) mc_st_v4(comm.mc + eoff, o);                 // one store, delivered to every GPU by the switch
    else {
      for (int p = 0; p < comm.world; ++p) st_global_v4(comm.heap[p] + eoff, o);
    }
  }
  __threadfence_system();
  block_barrier(comm, ep);          // my copy of C is complete once every rank's CTA b has finished multicasting
  epoch_store(comm, ep);
}

// ===================================================================================================
// CTA-pair (cta_group::2) variant of the TN GEMM / implicit-GEMM convolution: two SMs of one TPC form a cluster and
// execute ONE tcgen05.mma of M = 256: each CTA stages its own 128 rows of A and HALF of the B tile (N/2 rows), the
// leader's single thread issues the MMA for both, and each CTA's TMEM receives its 128 accumulator rows.  Per SM and
// k-block this moves 16 KB (A) + BN/2 x 128 B (B) for 128 x BN x 64 MACs — a third less L2->SM traffic than the 1-CTA
// kernel at BN = 256, and half the shared-memory operand reads per MMA (the N = 64 / 128 layers stop being smem-bound).
//   full_bar   (leader's)  <- TMA complete_tx from BOTH CTAs (cp.async.bulk.tensor...cta_group::2, peer bit cleared)
//   empty_bar  (each CTA)  <- tcgen05.commit.cta_group::2 ... multicast::cluster (mask 0b11)
//   tmem_full  (each CTA)  <- same multicast commit after the last k-block
//   tmem_empty (leader's)  <- remote mbarrier.arrive from both CTAs' epilogue threads
// ===================================================================================================
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;     // shared::cluster address of the even (leader) CTA of the pair
constexpr uint64_t kCacheHintNormal = 0x1000000000000000ull;

DEVI uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
DEVI void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
DEVI void tma_load_2d_2sm(void* smem_dst, const void* tmap, uint64_t* leader_bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
               ::"r"(smem_u32(smem_dst)), "l"((uint64_t)tmap), "r"(smem_u32(leader_bar) & kPeerBitMask), "r"(c0), "r"(c1), "l"(kCacheHintNormal) : "memory");
}
DEVI void tma_load_im2col_4d_2sm(void* smem_dst, const void* tmap, uint64_t* leader_bar, int c, int w, int h, int n, uint16_t off_w, uint16_t off_h) {
  asm volatile("cp.async.bulk.tensor.4d.im2col.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
               " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8}, %9;"
               ::"r"(smem_u32(smem_dst)), "l"((uint64_t)tmap), "r"(smem_u32(leader_bar) & kPeerBitMask), "r"(c), "r"(w), "r"(h), "r"(n),
                 "h"(off_w), "h"(off_h), "l"(kCacheHintNormal) : "memory");
}
DEVI void tma_load_3d_2sm(void* smem_dst, const void* tmap, uint64_t* leader_bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
               ::"r"(smem_u32(smem_dst)), "l"((uint64_t)tmap), "r"(smem_u32(leader_bar) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "l"(kCacheHintNormal) : "memory");
}
DEVI void umma_bf16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  const uint32_t z = 0;
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}"
               ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(z) : "memory");
}
DEVI void umma_commit_2sm(uint64_t* bar) {           // arrives on `bar` in BOTH CTAs of the pair
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
DEVI void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
template <int NCOLS> DEVI void tmem_alloc_2sm(uint32_t* dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(NCOLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int NCOLS> DEVI void tmem_dealloc_2sm(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}

template <int BN> struct Cfg2 {
  static constexpr int kABytes = BM * BK * 2;                 // this CTA's 128 rows of A
  static constexpr int kBBytes = (BN / 2) * BK * 2;           // this CTA's half of the B tile
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kCBytes = BM * kEpiChunk * 2;
  static constexpr int kBudget = 227 * 1024 - 1024 - 256 - 512;
  static constexpr int kStages = ((kBudget - 2 * kCBytes) / kStageBytes) > 8 ? 8 : ((kBudget - 2 * kCBytes) / kStageBytes);
  static constexpr int kTmemCols = 2 * BN < 32 ? 32 : 2 * BN;
  static constexpr int kSmemBytes = kStages * kStageBytes + 2 * kCBytes + 1024 + 256;
};

template <int BN, bool kStats, bool kConv, bool kBMN = false, bool kDirect = false>     // kDirect: see gemm_bf16_tn_kernel
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreadsTN, 1)
gemm_bf16_tn_2cta_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                         const __grid_constant__ CUtensorMap tmap_c, int M, int N, int K, float* __restrict__ stats, const ConvGeom geom,
                         __nv_bfloat16* __restrict__ c_ptr = nullptr, int ldc = 0) {
  using C = Cfg2<BN>;
  constexpr int BM2 = 2 * BM;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + C::kStages * C::kABytes;
  uint8_t* smem_c = smem + C::kStages * C::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_c + 2 * C::kCBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + C::kStages;
  uint64_t* tmem_full = bars + 2 * C::kStages;
  uint64_t* tmem_empty = bars + 2 * C::kStages + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * C::kStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int num_m = (M + BM2 - 1) / BM2, num_n = (N + BN - 1) / BN, num_k = (K + BK - 1) / BK;
  const int num_tiles = num_m * num_n;
  int t_first, t_stride;
  tile_walk<kStats>(pair, num_pairs, num_n, num_tiles, t_first, t_stride);
  constexpr int kChunks = BN / kEpiChunk;
  constexpr int kActiveGroups = kChunks < kEpiGroups ? kChunks : kEpiGroups;

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmap_a); tma_prefetch_desc(&tmap_b); tma_prefetch_desc(&tmap_c); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 2 * kEpiThreads * kActiveGroups); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_2sm<C::kTmemCols>(tmem_ptr);
  tc_fence_before();
  cluster_sync_all();                 // both CTAs' barriers are initialised before any remote arrive / complete_tx
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs: own A rows, own half of B; bytes land on the leader's barrier) ====
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int t = t_first; t < num_tiles; t += t_stride) {
        int m_blk, n_blk; map_tile<kStats>(t, num_m, num_n, m_blk, n_blk);
        const int m0 = m_blk * BM2 + (int)rank * BM;
        int cn = 0, ch = 0, cw = 0;
        if constexpr (kConv) {
          const int pq = geom.P * geom.Q;
          cn = m0 / pq; const int rem = m0 - cn * pq, p0 = rem / geom.Q;
          ch = geom.lower + geom.stride * p0; cw = geom.lower + geom.stride * (rem - p0 * geom.Q);
        }
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (leader) mbar_expect_tx(&full_bar[stage], 2u * C::kStageBytes);
          if constexpr (kConv) {
            const int tap = kb / geom.cblocks, cb = kb - tap * geom.cblocks, r = tap / geom.S, sx = tap - r * geom.S;
            tma_load_im2col_4d_2sm(smem_a + stage * C::kABytes, &tmap_a, &full_bar[stage], cb * 64, cw, ch, cn, (uint16_t)sx, (uint16_t)r);
          } else {
            tma_load_2d_2sm(smem_a + stage * C::kABytes, &tmap_a, &full_bar[stage], kb * BK, m0);
          }
          if constexpr (kBMN) {
            // B = W[K, N] row-major (dgrad): this CTA's half of the N range as 64-wide MN-major slabs
            const int nb0 = n_blk * BN + (int)rank * (BN / 2);
#pragma unroll
            for (int sl = 0; sl < BN / 128; ++sl) {
              if constexpr (kConv) {
                const int tap = kb / geom.cblocks, cb = kb - tap * geom.cblocks;
                tma_load_3d_2sm(smem_b + stage * C::kBBytes + sl * kSlabBytes, &tmap_b, &full_bar[stage], nb0 + sl * 64,
                                geom.flip ? geom.taps - 1 - tap : tap, cb * 64);
              } else {
                tma_load_2d_2sm(smem_b + stage * C::kBBytes + sl * kSlabBytes, &tmap_b, &full_bar[stage], nb0 + sl * 64, kb * BK);
              }
            }
          } else {
            tma_load_2d_2sm(smem_b + stage * C::kBBytes, &tmap_b, &full_bar[stage], kb * BK, n_blk * BN + (int)rank * (BN / 2));
          }
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: leader CTA only, one thread, M = 256 across the pair =====================
    if (leader && elect_one()) {
      constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((kBMN ? 1u : 0u) << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM2 >> 4) << 24);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int t = t_first; t < num_tiles; t += t_stride) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);       // both CTAs' epilogues have drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&full_bar[stage], phase);             // bytes of BOTH CTAs have landed
          tc_fence_after();
          const uint64_t adesc = make_kmajor_sw128_desc(smem_a + stage * C::kABytes);
          const uint64_t bdesc = kBMN ? make_mnmajor_sw128_desc(smem_b + stage * C::kBBytes, kSlabBytes)
                                      : make_kmajor_sw128_desc(smem_b + stage * C::kBBytes);
          constexpr uint64_t kBStep = kBMN ? (UK * 128 >> 4) : (UK * 2 >> 4);
#pragma unroll
          for (int k = 0; k < BK / UK; ++k)
            umma_bf16_2sm(d_tmem, adesc + (uint64_t)(k * UK * 2 >> 4), bdesc + (uint64_t)k * kBStep, idesc, (kb | k) != 0);
          umma_commit_2sm(&empty_bar[stage]);             // frees the stage in both CTAs
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit_2sm(&tmem_full[acc]);                 // publishes the accumulator to both epilogues
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue: each CTA drains its own 128 accumulator rows =====================
    const int grp = (warp - 4) >> 2;
    if (grp < kChunks) {
      const int ew = warp & 3, et = threadIdx.x - 128 - grp * 128;
      const int row = ew * 32 + lane;
      const bool issuer = et == 0;
      const int bar_a = 1 + 2 * grp, bar_b = 2 + 2 * grp;
      uint8_t* cbuf = smem_c + grp * C::kCBytes;
      int acc = 0; uint32_t acc_phase = 0;
      constexpr int kMyChunks = (kChunks + kEpiGroups - 1) / kEpiGroups;
      float st[kMyChunks][4];
#pragma unroll
      for (int c = 0; c < kMyChunks; ++c) { st[c][0] = st[c][1] = st[c][2] = st[c][3] = 0.f; }
      int cur_n = -1;
      auto flush_stats = [&](int n_blk) {
        if (!kStats || n_blk < 0) return;
        const int wcol = et & 31;
#pragma unroll
        for (int ci = 0; ci < kMyChunks; ++ci) {
          const int c = grp + ci * kEpiGroups;
          if (c < kChunks) {
            const int col = n_blk * BN + c * kEpiChunk + 2 * wcol;
            if (col < N) { atomicAdd(&stats[col], st[ci][0]); atomicAdd(&stats[N + col], st[ci][2]); }
            if (col + 1 < N) { atomicAdd(&stats[col + 1], st[ci][1]); atomicAdd(&stats[N + col + 1], st[ci][3]); }
          }
          st[ci][0] = st[ci][1] = st[ci][2] = st[ci][3] = 0.f;
        }
      };
      for (int t = t_first; t < num_tiles; t += t_stride) {
        int m_blk, n_blk; map_tile<kStats>(t, num_m, num_n, m_blk, n_blk);
        const int m0 = m_blk * BM2 + (int)rank * BM;
        if (kStats && n_blk != cur_n) { flush_stats(cur_n); cur_n = n_blk; }
        mbar_wait(&tmem_full[acc], acc_phase);
        tc_fence_after();
        const uint32_t tbase = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * BN);
        uint32_t v[2][32];
        tmem_ld32(tbase + grp * kEpiChunk, v[0]);
        tmem_ld32(tbase + grp * kEpiChunk + 32, v[1]);
#pragma unroll
        for (int ci = 0; ci < kMyChunks; ++ci) {
          const int c = grp + ci * kEpiGroups;
          if (c >= kChunks) break;
          tmem_ld_wait();
          const bool last = c + kEpiGroups >= kChunks;
          if (last) { tc_fence_before(); mbar_arrive_leader(&tmem_empty[acc]); }
          const int n0 = n_blk * BN + c * kEpiChunk;
          uint4 w[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float f[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(v[(q * 8 + i) >> 5][(q * 8 + i) & 31]);
            w[q] = make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
          }
          if (!last) {
            tmem_ld32(tbase + (c + kEpiGroups) * kEpiChunk, v[0]);
            tmem_ld32(tbase + (c + kEpiGroups) * kEpiChunk + 32, v[1]);
          }
          if constexpr (!kDirect) { if (issuer) tma_store_wait_read<0>(); }
          named_bar_sync(bar_a, kEpiThreads);
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<uint4*>(cbuf + row * 128 + ((q ^ (row & 7)) << 4)) = w[q];
          if constexpr (!kDirect) fence_proxy_async_smem();
          named_bar_sync(bar_b, kEpiThreads);
          if constexpr (kDirect) {
            const int sub = et & 7, rr = et >> 3;
            if (n0 + sub * 8 < N) {
#pragma unroll
              for (int p = 0; p < 8; ++p) {
                const int r = p * 16 + rr;
                if (m0 + r < M)
                  st_global_v4(c_ptr + (size_t)(m0 + r) * (size_t)ldc + n0 + sub * 8,
                               *reinterpret_cast<const uint4*>(cbuf + r * 128 + ((sub ^ (r & 7)) << 4)));
              }
            }
          } else {
            if (issuer) { tma_store_2d(&tmap_c, cbuf, n0, m0); tma_store_commit(); }
          }
          if (kStats) {
            const int wcol = et & 31, rgrp = et >> 5;
            const int q = wcol >> 2, wi = wcol & 3;
            const int rows_valid = M - m0;
            float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll 8
            for (int r = rgrp * 32; r < rgrp * 32 + 32; ++r) {
              const uint32_t wv = *reinterpret_cast<const uint32_t*>(cbuf + r * 128 + ((q ^ (r & 7)) << 4) + wi * 4);
              const float a = __uint_as_float(wv << 16), b = __uint_as_float(wv & 0xffff0000u);
              if (r < rows_valid) { s0 += a; s1 += b; q0 = fmaf(a, a, q0); q1 = fmaf(b, b, q1); }
            }
            st[ci][0] += s0; st[ci][1] += s1; st[ci][2] += q0; st[ci][3] += q1;
          }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      flush_stats(cur_n);
      if constexpr (!kDirect) { if (issuer) tma_store_wait_all(); }
    }
  }
  tc_fence_before();
  cluster_sync_all();                 // the peer's smem / TMEM stay alive until every MMA and epilogue of the pair is done
  if (warp == 2) { tc_fence_after(); tmem_dealloc_2sm<C::kTmemCols>(tmem_base); }
}

// ---- host side ------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
// cuTensorMapEncode* is a driver entry point and needs a context current on the CALLING thread.  A thread that has made no runtime call
// yet has none — e.g. PyTorch's autograd thread when the first thing a backward does is one of our GEMMs with its output served from the
// caching allocator (seen as error 201 in tests/test_gpu_gemm.py when that file runs alone).  On that error: make the device that owns the
// operand current (the runtime then binds its primary context to this thread) and encode again.
bool bind_context_of(const void* ptr) {
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess || a.type != cudaMemoryTypeDevice) { cudaGetLastError(); return false; }
  return cudaSetDevice(a.device) == cudaSuccess && cudaFree(nullptr) == cudaSuccess;
}
#define ENC_RETRY(call, ptr) ({ CUresult _r = (call); if (_r == CUDA_ERROR_INVALID_CONTEXT && bind_context_of(ptr)) _r = (call); _r; })
std::atomic<unsigned long long> g_launches{0};
thread_local char g_err[256];

bool load_encode() {
  if (g_encode) return true;
  void* fn = nullptr; cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) return false;
  g_encode = (EncodeTiledFn)fn;
  return true;
}

// SHIPYARD_GEMM_DIRECT_STORE=1 selects the kDirect epilogue (st.global instead of TMA stores) in the TN / CTA-pair GEMM and
// im2col convolution launches; off by default (measured in round 2: no gain on the whole step).
bool direct_store() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("SHIPYARD_GEMM_DIRECT_STORE"); v = (e && e[0] && e[0] != '0') ? 1 : 0; }
  return v == 1;
}

bool epi_alt() {                      // SHIPYARD_GEMM_EPI_ALT=1 (with SHIPYARD_GEMM_DIRECT_STORE=1): alternate-tile epilogue for 64-column GEMM tiles
  static int v = -1;
  if (v < 0) { const char* e = getenv("SHIPYARD_GEMM_EPI_ALT"); v = (e && e[0] && e[0] != '0') ? 1 : 0; }
  return v == 1;
}

// 2D bf16 tensor map: dims {inner, outer}, row pitch `ld` elements, box {box_inner, box_outer}, 128B swizzle
bool make_map(CUtensorMap* m, const void* ptr, uint64_t inner, uint64_t outer, uint64_t ld, uint32_t box_inner, uint32_t box_outer) {
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = ENC_RETRY(g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE), ptr);
  if (r != CUDA_SUCCESS) { snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled failed (%d)", (int)r); return false; }
  return true;
}

typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const int*,
                                   const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeIm2colFn g_encode_im2col = nullptr;
bool load_encode_im2col() {
  if (g_encode_im2col) return true;
  void* fn = nullptr; cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) return false;
  g_encode_im2col = (EncodeIm2colFn)fn;
  return true;
}
// NHWC bf16 activation [N, H, W, C] as an im2col tensor map: box = 128 pixels x 64 channels, filter extent (R, S), padding `pad`
bool make_im2col_map(CUtensorMap* m, const void* ptr, int N, int H, int W, int C, int R, int S, int pad, int stride, uint32_t pixels) {
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  int lower[2] = {-pad, -pad};
  int upper[2] = {pad - (S - 1), pad - (R - 1)};
  cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  CUresult r = ENC_RETRY(g_encode_im2col(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, lower, upper, 64, pixels, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE), ptr);
  if (r != CUDA_SUCCESS) { snprintf(g_err, sizeof g_err, "cuTensorMapEncodeIm2col failed (%d)", (int)r); return false; }
  return true;
}
// weights [Cout][taps][Cin] as a 3D map {Cin, taps, Cout}, box {64, 1, 64}: one MN-major slab (64 co-rows x 64 ci) per load
bool make_w3d_map(CUtensorMap* m, const void* ptr, int Cout, int taps, int Cin) {
  cuuint64_t dims[3] = {(cuuint64_t)Cin, (cuuint64_t)taps, (cuuint64_t)Cout};
  cuuint64_t strides[2] = {(cuuint64_t)Cin * 2, (cuuint64_t)taps * Cin * 2};
  cuuint32_t box[3] = {64, 1, 64};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = ENC_RETRY(g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE), ptr);
  if (r != CUDA_SUCCESS) { snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled(3D) failed (%d)", (int)r); return false; }
  return true;
}

// Implicit-GEMM convolution launch.  dgrad == false: y[N,P,Q,Co] = conv(x[N,H,W,Ci], w[Co,R,S,Ci]) (+BN statistics);
// dgrad == true (stride 1): x_grad[N,H,W,Ci] = conv(dy[N,P,Q,Co], rot180(w)^T), weights read in place as an MN-major operand.
template <int BN>
int launch_conv(const void* act, const void* wgt, void* out, int Nb, int H, int W, int Ca, int Cn, int R, int S, int pad, int stride,
                bool dgrad, float* stats, int max_ctas, cudaStream_t s) {
  using C = Cfg<BN>;
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  const int M = Nb * P * Q, N = Cn, K = R * S * Ca;
  CUtensorMap ta, tb, tc;
  if (!make_im2col_map(&ta, act, Nb, H, W, Ca, R, S, pad, stride, BM)) return 3;
  if (dgrad) { if (!make_w3d_map(&tb, wgt, Ca, R * S, Cn)) return 3; }        // wgt = W[Co = Ca][taps][Ci = Cn]
  else if (!make_map(&tb, wgt, K, N, K, BK, BN)) return 3;
  if (!make_map(&tc, out, N, M, N, kEpiChunk, BM)) return 3;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);
  int grid = tiles < sms ? tiles : sms;
  if (max_ctas > 0 && grid > max_ctas) grid = max_ctas;
  ConvGeom g{P, Q, S, R * S, Ca / 64, stride, -pad, dgrad ? 1 : 0};
  auto go = [&](auto kern) -> int {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes);
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "smem attribute: %s", cudaGetErrorString(e)); return 4; }
    kern<<<grid, kThreadsTN, C::kSmemBytes, s>>>(ta, tb, tc, M, N, K, (const __nv_bfloat16*)nullptr, stats, g, (__nv_bfloat16*)out, N, EpiAffine{});
    e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "launch: %s", cudaGetErrorString(e)); return 5; }
    g_launches.fetch_add(1);
    return 0;
  };
  if (direct_store() && N % 8 == 0) {
    if (dgrad) return go(gemm_bf16_tn_kernel<BN, false, false, true, true, true>);
    if (stats) return go(gemm_bf16_tn_kernel<BN, true, false, false, true, true>);
    return go(gemm_bf16_tn_kernel<BN, false, false, false, true, true>);
  }
  if (dgrad) return go(gemm_bf16_tn_kernel<BN, false, false, true, true>);
  if (stats) return go(gemm_bf16_tn_kernel<BN, true, false, false, true>);
  return go(gemm_bf16_tn_kernel<BN, false, false, false, true>);
}

template <int BN>
int launch(const void* A, const void* B, void* Cc, int M, int N, int K, int lda, int ldb, int ldc, const void* bias, float* stats,
           int max_ctas, cudaStream_t s, bool b_mn = false) {
  using C = Cfg<BN>;
  CUtensorMap ta, tb, tc;
  if (!make_map(&ta, A, K, M, lda, BK, BM) || !make_map(&tc, Cc, N, M, ldc, kEpiChunk, BM)) return 3;
  if (!(b_mn ? make_map(&tb, B, N, K, ldb, 64, BK) : make_map(&tb, B, K, N, ldb, BK, BN))) return 3;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);
  int grid = tiles < sms ? tiles : sms;
  if (max_ctas > 0 && grid > max_ctas) grid = max_ctas;
  auto go = [&](auto kern) -> int {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes);
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "smem attribute: %s", cudaGetErrorString(e)); return 4; }
    kern<<<grid, kThreadsTN, C::kSmemBytes, s>>>(ta, tb, tc, M, N, K, (const __nv_bfloat16*)bias, stats, ConvGeom{}, (__nv_bfloat16*)Cc, ldc,
                                                 EpiAffine{});
    e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "launch: %s", cudaGetErrorString(e)); return 5; }
    g_launches.fetch_add(1);
    return 0;
  };
  if (stats && bias) { snprintf(g_err, sizeof g_err, "stats and bias cannot be combined"); return 2; }
  const bool direct = direct_store() && N % 8 == 0;
  if constexpr (BN == 64) {
    if (direct && epi_alt() && !bias) {
      if (b_mn) {
        if (stats) { snprintf(g_err, sizeof g_err, "MN-major B: no fused epilogue"); return 2; }
        return go(gemm_bf16_tn_kernel<64, false, false, true, false, true, true>);
      }
      return stats ? go(gemm_bf16_tn_kernel<64, true, false, false, false, true, true>) : go(gemm_bf16_tn_kernel<64, false, false, false, false, true, true>);
    }
  }
  if (b_mn) {
    if (stats || bias) { snprintf(g_err, sizeof g_err, "MN-major B: no fused epilogue"); return 2; }
    return direct ? go(gemm_bf16_tn_kernel<BN, false, false, true, false, true>) : go(gemm_bf16_tn_kernel<BN, false, false, true>);
  }
  if (stats) return direct ? go(gemm_bf16_tn_kernel<BN, true, false, false, false, true>) : go(gemm_bf16_tn_kernel<BN, true, false>);
  if (bias) return go(gemm_bf16_tn_kernel<BN, false, true>);
  return direct ? go(gemm_bf16_tn_kernel<BN, false, false, false, false, true>) : go(gemm_bf16_tn_kernel<BN, false, false>);
}

// Folded-BN epilogue launches (kAffine): the plain GEMM (conv == false: A [M, K] row-major) or the TMA-im2col convolution.
template <int BN>
int launch_affine(bool conv, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, int M, int N, int K, const ConvGeom& g,
                  void* out, int ldc, const EpiAffine& aff, int max_ctas, cudaStream_t s) {
  using C = Cfg<BN>;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);
  int grid = tiles < sms ? tiles : sms;
  if (max_ctas > 0 && grid > max_ctas) grid = max_ctas;
  auto go = [&](auto kern) -> int {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes);
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "smem attribute: %s", cudaGetErrorString(e)); return 4; }
    kern<<<grid, kThreadsTN, C::kSmemBytes, s>>>(ta, tb, tc, M, N, K, (const __nv_bfloat16*)nullptr, (float*)nullptr, g, (__nv_bfloat16*)out,
                                                 ldc, aff);
    e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "launch: %s", cudaGetErrorString(e)); return 5; }
    g_launches.fetch_add(1);
    return 0;
  };
  return conv ? go(gemm_bf16_tn_kernel<BN, false, false, false, true, true, false, true>)
              : go(gemm_bf16_tn_kernel<BN, false, false, false, false, true, false, true>);
}

// Shared argument checks of the two affine entry points: N % 8 (whole 16-byte pieces), aligned scale / shift / residual, and an output
// that does not overlap the residual (a row's residual would be overwritten by another CTA before it is read).
bool affine_args_ok(const void* out, long out_rows, int ldc, const float* scale, const float* shift, const void* residual, int ldr, int N) {
  if (N % 8 || !scale || !shift || (((uintptr_t)scale | (uintptr_t)shift | (uintptr_t)residual) & 15) || (residual && (ldr & 7))) {
    snprintf(g_err, sizeof g_err, "affine epilogue: N %% 8, 16-byte aligned scale / shift / residual, residual pitch %% 8"); return false;
  }
  if (residual) {
    const uintptr_t o0 = (uintptr_t)out, o1 = o0 + (uintptr_t)out_rows * ldc * 2;
    const uintptr_t r0 = (uintptr_t)residual, r1 = r0 + (uintptr_t)out_rows * ldr * 2;
    if (o0 < r1 && r0 < o1) { snprintf(g_err, sizeof g_err, "affine epilogue: out must not alias residual"); return false; }
  }
  return true;
}

}  // namespace

#include "conv_halo.inc"
#include "wgrad_halo.inc"
#include "stem_s2d.inc"

extern "C" const char* sy_gemm_last_error() { return g_err; }
extern "C" unsigned long long sy_gemm_launch_count() { return g_launches.load(); }

// C[M,N] = A[M,K] * B[N,K]^T (+bias) ; bf16 in/out, fp32 accumulate in TMEM.  lda/ldb/ldc in elements.
// stats (optional): float[2*N], caller-zeroed: per-column sum and sum of squares of the bf16 output.
// Requirements: pointers 16B aligned, lda/ldb/ldc multiples of 8, K >= 1.
extern "C" int sy_gemm_bf16_tn(const void* A, const void* B, void* C, int M, int N, int K, int lda, int ldb, int ldc,
                               const void* bias, float* stats, int block_n, int max_ctas, void* stream) {
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  if ((lda | ldb | ldc) & 7 || ((uintptr_t)A | (uintptr_t)B | (uintptr_t)C) & 15) {
    snprintf(g_err, sizeof g_err, "alignment: pointers must be 16B aligned and leading dimensions multiples of 8");
    return 1;
  }
  if (!load_encode()) { snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled unavailable (no driver?)"); return 6; }
  cudaStream_t s = (cudaStream_t)stream;
  if (block_n <= 0) block_n = N > 128 ? 256 : (N > 64 ? 128 : 64);
  switch (block_n) {
    case 64: return launch<64>(A, B, C, M, N, K, lda, ldb, ldc, bias, stats, max_ctas, s);
    case 128: return launch<128>(A, B, C, M, N, K, lda, ldb, ldc, bias, stats, max_ctas, s);
    case 256: return launch<256>(A, B, C, M, N, K, lda, ldb, ldc, bias, stats, max_ctas, s);
  }
  snprintf(g_err, sizeof g_err, "block_n must be 64, 128 or 256");
  return 1;
}

// CTA-pair launches.  Requirements on top of the 1-CTA entry points: N %% block_n == 0 (each CTA loads exactly half a B tile).
// mode 0: B K-major [N, K]; mode 1: B = W[K, N] row-major (MN-major operand, dgrad of a 1x1 conv / Linear);
// mode 2: conv dgrad, B = W[Cout][taps][Cin] through the 3-D map.
template <int BN>
int launch_2cta(bool conv, int bmode, const void* A, const void* B, void* Cc, int M, int N, int K, int lda, int ldb, int ldc, float* stats,
                const ConvGeom& g, const int* im2col /* Nb,H,W,C,R,S,pad,stride or null */, int max_ctas, cudaStream_t s) {
  using C = Cfg2<BN>;
  CUtensorMap ta, tb, tc;
  if (conv) { if (!make_im2col_map(&ta, A, im2col[0], im2col[1], im2col[2], im2col[3], im2col[4], im2col[5], im2col[6], im2col[7], BM)) return 3; }
  else if (!make_map(&ta, A, K, M, lda, BK, BM)) return 3;
  if (bmode == 0) { if (!make_map(&tb, B, K, N, ldb, BK, BN / 2)) return 3; }
  else if (bmode == 1) { if (!make_map(&tb, B, N, K, ldb, 64, BK)) return 3; }
  else if (!make_w3d_map(&tb, B, im2col[3], im2col[4] * im2col[5], N)) return 3;       // W[Co = act channels][taps][Ci = N]
  if (!make_map(&tc, Cc, N, M, ldc, kEpiChunk, BM)) return 3;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int tiles = ((M + 2 * BM - 1) / (2 * BM)) * (N / BN);
  int pairs = tiles < sms / 2 ? tiles : sms / 2;
  if (max_ctas > 1 && pairs > max_ctas / 2) pairs = max_ctas / 2;
  auto go = [&](auto kern) -> int {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes);
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "smem attribute: %s", cudaGetErrorString(e)); return 4; }
    kern<<<2 * pairs, kThreadsTN, C::kSmemBytes, s>>>(ta, tb, tc, M, N, K, stats, g, (__nv_bfloat16*)Cc, ldc);
    e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "launch: %s", cudaGetErrorString(e)); return 5; }
    g_launches.fetch_add(1);
    return 0;
  };
  if (direct_store()) {            // N % block_n == 0 here, so every 16-byte piece is whole
    if (bmode != 0) {
      if (stats) { snprintf(g_err, sizeof g_err, "2-CTA dgrad: no fused statistics"); return 2; }
      return conv ? go(gemm_bf16_tn_2cta_kernel<BN, false, true, true, true>) : go(gemm_bf16_tn_2cta_kernel<BN, false, false, true, true>);
    }
    if (conv) return stats ? go(gemm_bf16_tn_2cta_kernel<BN, true, true, false, true>) : go(gemm_bf16_tn_2cta_kernel<BN, false, true, false, true>);
    return stats ? go(gemm_bf16_tn_2cta_kernel<BN, true, false, false, true>) : go(gemm_bf16_tn_2cta_kernel<BN, false, false, false, true>);
  }
  if (bmode != 0) {
    if (stats) { snprintf(g_err, sizeof g_err, "2-CTA dgrad: no fused statistics"); return 2; }
    return conv ? go(gemm_bf16_tn_2cta_kernel<BN, false, true, true>) : go(gemm_bf16_tn_2cta_kernel<BN, false, false, true>);
  }
  if (conv) return stats ? go(gemm_bf16_tn_2cta_kernel<BN, true, true>) : go(gemm_bf16_tn_2cta_kernel<BN, false, true>);
  return stats ? go(gemm_bf16_tn_2cta_kernel<BN, true, false>) : go(gemm_bf16_tn_2cta_kernel<BN, false, false>);
}

extern "C" int sy_gemm_bf16_tn_2cta(const void* A, const void* B, void* C, int M, int N, int K, int lda, int ldb, int ldc, float* stats,
                                    int block_n, int max_ctas, int b_mn, void* stream) {
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  if ((lda | ldb | ldc) & 7 || ((uintptr_t)A | (uintptr_t)B | (uintptr_t)C) & 15) {
    snprintf(g_err, sizeof g_err, "alignment: pointers must be 16B aligned and leading dimensions multiples of 8"); return 1;
  }
  if (!load_encode()) { snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled unavailable (no driver?)"); return 6; }
  if (block_n <= 0) block_n = N % 256 == 0 ? 256 : (N % 128 == 0 ? 128 : 0);
  if (block_n == 0 || N % block_n) { snprintf(g_err, sizeof g_err, "2-CTA GEMM needs N %% block_n == 0 (block_n 128 or 256)"); return 1; }
  ConvGeom g{};
  switch (block_n) {
    case 128: return launch_2cta<128>(false, b_mn ? 1 : 0, A, B, C, M, N, K, lda, ldb, ldc, stats, g, nullptr, max_ctas, (cudaStream_t)stream);
    case 256: return launch_2cta<256>(false, b_mn ? 1 : 0, A, B, C, M, N, K, lda, ldb, ldc, stats, g, nullptr, max_ctas, (cudaStream_t)stream);
  }
  snprintf(g_err, sizeof g_err, "block_n must be 128 or 256");
  return 1;
}

// CTA-pair convolution.  dgrad == 0: out[N,P,Q,c_out] = conv(act[N,H,W,c_act], wgt[c_out,R,S,c_act]) (+BN statistics);
// dgrad == 1 (stride 1, 'same'): out[N,H,W,c_out] from act = dY[N,H,W,c_act], wgt = W[c_act,R,S,c_out] read in place.
// N*P*Q %% 256 == 0, c_out %% block_n == 0, c_act %% 64 == 0.
extern "C" int sy_conv_bf16_nhwc_2cta(const void* act, const void* wgt, void* out, int Nb, int H, int W, int c_act, int c_out, int R, int S,
                                      int pad, int stride, int dgrad, float* stats, int block_n, int max_ctas, void* stream) {
  if (c_act % 64 || ((uintptr_t)act | (uintptr_t)wgt | (uintptr_t)out) & 15) { snprintf(g_err, sizeof g_err, "conv: act channels %% 64, aligned tensors"); return 1; }
  if (dgrad && (stride != 1 || stats)) { snprintf(g_err, sizeof g_err, "conv dgrad: stride 1, no stats"); return 1; }
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  if (((long)Nb * P * Q) % (2 * BM)) { snprintf(g_err, sizeof g_err, "2-CTA conv: N*P*Q must be a multiple of 256"); return 1; }
  if (dgrad && (P != H || Q != W)) { snprintf(g_err, sizeof g_err, "conv dgrad: 'same' padding only"); return 1; }
  if (!load_encode() || !load_encode_im2col()) { snprintf(g_err, sizeof g_err, "cuTensorMapEncode* unavailable (no driver?)"); return 6; }
  if (block_n <= 0) block_n = c_out % 256 == 0 ? 256 : (c_out % 128 == 0 ? 128 : 0);
  if (block_n == 0 || c_out % block_n) { snprintf(g_err, sizeof g_err, "2-CTA conv needs out channels %% block_n == 0 (block_n 128 or 256)"); return 1; }
  const int M = Nb * P * Q, K = R * S * c_act;
  ConvGeom g{P, Q, S, R * S, c_act / 64, stride, -pad, dgrad ? 1 : 0};
  const int geo[8] = {Nb, H, W, c_act, R, S, pad, stride};
  const int bmode = dgrad ? 2 : 0;
  switch (block_n) {
    case 128: return launch_2cta<128>(true, bmode, act, wgt, out, M, c_out, K, 0, K, c_out, stats, g, geo, max_ctas, (cudaStream_t)stream);
    case 256: return launch_2cta<256>(true, bmode, act, wgt, out, M, c_out, K, 0, K, c_out, stats, g, geo, max_ctas, (cudaStream_t)stream);
  }
  snprintf(g_err, sizeof g_err, "block_n must be 128 or 256");
  return 1;
}

// Convolution as implicit GEMM on tcgen05 with TMA im2col loads (no im2col buffer, padding by TMA zero fill).
//   dgrad == 0: out[N,P,Q,Cout] = conv(act[N,H,W,Cin], wgt[Cout,R,S,Cin]), optional BN statistics of `out` in stats[2*Cout]
//   dgrad == 1: out[N,H,W,Cin]  = dgrad of the same convolution from act = dY[N,P,Q,Cout] (stride 1 only); wgt as above
// c_act = channels of `act`, c_out = channels of `out`.  Requirements: channels of `act` %% 64 == 0, c_out %% 8 == 0,
// N*P*Q %% 128 == 0 (whole M tiles), tensors dense NHWC / KRSC and 16-byte aligned.
extern "C" int sy_conv_bf16_nhwc(const void* act, const void* wgt, void* out, int Nb, int H, int W, int c_act, int c_out, int R, int S,
                                 int pad, int stride, int dgrad, float* stats, int block_n, int max_ctas, void* stream) {
  if (c_act % 64 || c_out % 8 || ((uintptr_t)act | (uintptr_t)wgt | (uintptr_t)out) & 15) {
    snprintf(g_err, sizeof g_err, "conv: act channels %% 64, out channels %% 8, 16B aligned tensors"); return 1;
  }
  if (dgrad && (stride != 1 || stats)) { snprintf(g_err, sizeof g_err, "conv dgrad: stride 1, no stats"); return 1; }
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  if (((long)Nb * P * Q) % BM) { snprintf(g_err, sizeof g_err, "conv: N*P*Q must be a multiple of 128"); return 1; }
  if (dgrad && (P != H || Q != W)) { snprintf(g_err, sizeof g_err, "conv dgrad: 'same' padding only"); return 1; }
  if (!load_encode() || !load_encode_im2col()) { snprintf(g_err, sizeof g_err, "cuTensorMapEncode* unavailable (no driver?)"); return 6; }
  cudaStream_t s = (cudaStream_t)stream;
  if (block_n <= 0) block_n = c_out > 128 ? 256 : (c_out > 64 ? 128 : 64);
  switch (block_n) {
    case 64: return launch_conv<64>(act, wgt, out, Nb, H, W, c_act, c_out, R, S, pad, stride, dgrad != 0, stats, max_ctas, s);
    case 128: return launch_conv<128>(act, wgt, out, Nb, H, W, c_act, c_out, R, S, pad, stride, dgrad != 0, stats, max_ctas, s);
    case 256: return launch_conv<256>(act, wgt, out, Nb, H, W, c_act, c_out, R, S, pad, stride, dgrad != 0, stats, max_ctas, s);
  }
  snprintf(g_err, sizeof g_err, "block_n must be 64, 128 or 256");
  return 1;
}

// Inference GEMM with BatchNorm folded into the epilogue (1x1 / stride-1 convolution on NHWC activations):
//   C[m, n] = act(sum_k A[m, k] * B[n, k] * scale[n] + shift[n] (+ residual[m * ldr + n]))
// act = ReLU when relu != 0, else identity; scale / shift fp32[N]; residual bf16 or null, and it must not overlap C.
// Requirements: those of sy_gemm_bf16_tn, N %% 8 == 0, scale / shift / residual 16-byte aligned, ldr %% 8 == 0.  block_n 64, 128 or 256.
extern "C" int sy_gemm_bf16_tn_affine(const void* A, const void* B, void* C, int M, int N, int K, int lda, int ldb, int ldc,
                                      const float* scale, const float* shift, const void* residual, int ldr, int relu, int block_n,
                                      int max_ctas, void* stream) {
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  if ((lda | ldb | ldc) & 7 || ((uintptr_t)A | (uintptr_t)B | (uintptr_t)C) & 15) {
    snprintf(g_err, sizeof g_err, "alignment: pointers must be 16B aligned and leading dimensions multiples of 8");
    return 1;
  }
  if (!affine_args_ok(C, M, ldc, scale, shift, residual, ldr, N)) return 1;
  if (!load_encode()) { snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled unavailable (no driver?)"); return 6; }
  if (block_n <= 0) block_n = N > 128 ? 256 : (N > 64 ? 128 : 64);
  CUtensorMap ta, tb, tc;
  if (!make_map(&ta, A, K, M, lda, BK, BM) || !make_map(&tc, C, N, M, ldc, kEpiChunk, BM)) return 3;
  const EpiAffine aff{scale, shift, (const __nv_bfloat16*)residual, ldr, relu ? 1 : 0};
  const ConvGeom g{};
  cudaStream_t s = (cudaStream_t)stream;
  switch (block_n) {
    case 64: if (!make_map(&tb, B, K, N, ldb, BK, 64)) return 3; return launch_affine<64>(false, ta, tb, tc, M, N, K, g, C, ldc, aff, max_ctas, s);
    case 128: if (!make_map(&tb, B, K, N, ldb, BK, 128)) return 3; return launch_affine<128>(false, ta, tb, tc, M, N, K, g, C, ldc, aff, max_ctas, s);
    case 256: if (!make_map(&tb, B, K, N, ldb, BK, 256)) return 3; return launch_affine<256>(false, ta, tb, tc, M, N, K, g, C, ldc, aff, max_ctas, s);
  }
  snprintf(g_err, sizeof g_err, "block_n must be 64, 128 or 256");
  return 1;
}

// Inference convolution with BatchNorm folded into the epilogue (TMA im2col implicit GEMM, 1-CTA):
//   out[N,P,Q,c_out] = act(conv(act_in[N,H,W,c_act], wgt[c_out,R,S,c_act]) * scale + shift (+ residual[N,P,Q,c_out]))
// Requirements: those of sy_conv_bf16_nhwc (c_act %% 64, c_out %% 8, N*P*Q %% 128), scale / shift / residual 16-byte aligned,
// residual dense NHWC like `out` and not overlapping it.
extern "C" int sy_conv_bf16_nhwc_affine(const void* act, const void* wgt, void* out, int Nb, int H, int W, int c_act, int c_out, int R, int S,
                                        int pad, int stride, const float* scale, const float* shift, const void* residual, int relu,
                                        int block_n, int max_ctas, void* stream) {
  if (c_act % 64 || c_out % 8 || ((uintptr_t)act | (uintptr_t)wgt | (uintptr_t)out) & 15) {
    snprintf(g_err, sizeof g_err, "conv: act channels %% 64, out channels %% 8, 16B aligned tensors"); return 1;
  }
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  if (((long)Nb * P * Q) % BM) { snprintf(g_err, sizeof g_err, "conv: N*P*Q must be a multiple of 128"); return 1; }
  const int M = Nb * P * Q, N = c_out, K = R * S * c_act;
  if (!affine_args_ok(out, M, N, scale, shift, residual, N, N)) return 1;
  if (!load_encode() || !load_encode_im2col()) { snprintf(g_err, sizeof g_err, "cuTensorMapEncode* unavailable (no driver?)"); return 6; }
  if (block_n <= 0) block_n = c_out > 128 ? 256 : (c_out > 64 ? 128 : 64);
  CUtensorMap ta, tb, tc;
  if (!make_im2col_map(&ta, act, Nb, H, W, c_act, R, S, pad, stride, BM) || !make_map(&tc, out, N, M, N, kEpiChunk, BM)) return 3;
  const EpiAffine aff{scale, shift, (const __nv_bfloat16*)residual, N, relu ? 1 : 0};
  const ConvGeom g{P, Q, S, R * S, c_act / 64, stride, -pad, 0};
  cudaStream_t s = (cudaStream_t)stream;
  switch (block_n) {
    case 64: if (!make_map(&tb, wgt, K, N, K, BK, 64)) return 3; return launch_affine<64>(true, ta, tb, tc, M, N, K, g, out, N, aff, max_ctas, s);
    case 128: if (!make_map(&tb, wgt, K, N, K, BK, 128)) return 3; return launch_affine<128>(true, ta, tb, tc, M, N, K, g, out, N, aff, max_ctas, s);
    case 256: if (!make_map(&tb, wgt, K, N, K, BK, 256)) return 3; return launch_affine<256>(true, ta, tb, tc, M, N, K, g, out, N, aff, max_ctas, s);
  }
  snprintf(g_err, sizeof g_err, "block_n must be 64, 128 or 256");
  return 1;
}

// Convolution weight gradient: dW[Cout][R][S][Cin] (+)= sum over output pixels of dY[pix][Cout] * im2col(x)[pix][(r,s,Cin)].
// One split-K launch covers every filter tap (work item = (tap, tile, K-split)).  ws: float[R*S*Cin*Cout], tickets:
// int[R*S*tiles]; both zero on entry and on exit.  Requirements: Cin %% 64, Cout %% 8, N*P*Q %% 128.
extern "C" int sy_conv_bf16_wgrad(const void* x, const void* dy, void* dw, int Nb, int H, int W, int Cin, int Cout, int R, int S, int pad,
                                  int stride, float* ws, int* tickets, int accumulate, int block_n, int splits, void* stream) {
  if (Cin % 64 || Cout % 8 || ((uintptr_t)x | (uintptr_t)dy) & 15 || ((uintptr_t)dw & 7)) {
    snprintf(g_err, sizeof g_err, "conv wgrad: Cin %% 64, Cout %% 8, aligned tensors"); return 1;
  }
  const int P = (H + 2 * pad - R) / stride + 1, Q = (W + 2 * pad - S) / stride + 1;
  const long Kl = (long)Nb * P * Q;
  if (Kl % BM) { snprintf(g_err, sizeof g_err, "conv wgrad: N*P*Q must be a multiple of 128"); return 1; }
  if (!load_encode() || !load_encode_im2col()) { snprintf(g_err, sizeof g_err, "cuTensorMapEncode* unavailable (no driver?)"); return 6; }
  const int taps = R * S, I = taps * Cin, J = Cout, K = (int)Kl;       // I index = tap * Cin + ci = the KRSC row of dW
  if (block_n <= 0) block_n = J > 128 ? 256 : (J > 64 ? 128 : 64);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaStream_t s = (cudaStream_t)stream;
  auto go = [&](auto kern, int BN, int smem) -> int {
    CUtensorMap ta, tb;
    if (!make_im2col_map(&ta, x, Nb, H, W, Cin, R, S, pad, stride, 64) || !make_map(&tb, dy, J, K, J, 64, BK)) return 3;
    const int tiles = ((I + BM - 1) / BM) * ((J + BN - 1) / BN), num_k = (K + BK - 1) / BK;
    int sp = splits;
    if (sp <= 0) { sp = sms / tiles; if (sp > num_k / 4) sp = num_k / 4; }     // floor: tiles * sp <= #SMs, a single wave
    if (sp < 1) sp = 1;
    if (sp > num_k) sp = num_k;
    if (sp > 1 && (!ws || !tickets)) { snprintf(g_err, sizeof g_err, "split-K needs a workspace"); return 2; }
    const long items = (long)tiles * sp;
    const int grid = (int)(items < sms ? items : sms);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "smem attribute: %s", cudaGetErrorString(e)); return 4; }
    ConvGeom g{P, Q, S, taps, Cin / 64, stride, -pad, 0};
    kern<<<grid, kThreads, smem, s>>>(ta, tb, I, J, K, sp, ws, tickets, (__nv_bfloat16*)dw, I, accumulate, g);
    e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "launch: %s", cudaGetErrorString(e)); return 5; }
    g_launches.fetch_add(1);
    return 0;
  };
  switch (block_n) {
    case 64: return go(gemm_bf16_nt_splitk_kernel<64, true>, 64, Cfg<64>::kSmemBytes);
    case 128: return go(gemm_bf16_nt_splitk_kernel<128, true>, 128, Cfg<128>::kSmemBytes);
    case 256: return go(gemm_bf16_nt_splitk_kernel<256, true>, 256, Cfg<256>::kSmemBytes);
  }
  snprintf(g_err, sizeof g_err, "block_n must be 64, 128 or 256");
  return 1;
}

// K10 v2: out (bf16 [M,N], symmetric, dense) = sum over ranks of A_r x B_r^T.  inbox: symmetric bf16 scratch of
// world * rows_per_rank * N elements, rows_per_rank = ceil(ceil(M/128) / world) * 128 (returned through *rows_per_rank_out
// when the pointers are null, so callers can size it).
extern "C" int sy_gemm_bf16_tn_rsag(const void* comm_view, size_t comm_view_bytes, const void* A, const void* B, size_t inbox_off,
                                    size_t out_off, int M, int N, int K, int lda, int ldb, int block_n, int* rows_per_rank_out, void* stream) {
  if (comm_view_bytes != sizeof(CommDev)) { snprintf(g_err, sizeof g_err, "communicator view size mismatch"); return 1; }
  CommDev cd; memcpy(&cd, comm_view, sizeof cd);
  const int num_m = (M + BM - 1) / BM;
  const int rpr = ((num_m + cd.world - 1) / cd.world) * BM;
  if (rows_per_rank_out) *rows_per_rank_out = rpr;
  if (!A || !B) return 0;                                    // size query
  if ((lda | ldb) & 7 || (N & 7) || ((uintptr_t)A | (uintptr_t)B) & 15 || ((inbox_off | out_off) & 15)) {
    snprintf(g_err, sizeof g_err, "alignment: A/B 16B aligned, lda/ldb/N %% 8, offsets %% 16"); return 1;
  }
  if (!load_encode()) { snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled unavailable"); return 6; }
  if (block_n <= 0) block_n = N > 128 ? 256 : (N > 64 ? 128 : 64);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaStream_t s = (cudaStream_t)stream;
  auto go = [&](auto kern, int BN, int smem) -> int {
    CUtensorMap ta, tb;
    if (!make_map(&ta, A, K, M, lda, BK, BM) || !make_map(&tb, B, K, N, ldb, BK, BN)) return 3;
    const int tiles = (rpr / BM) * cd.world * ((N + BN - 1) / BN);
    int grid = tiles < sms ? tiles : sms;
    if (grid > SY_MAX_BLOCKS) grid = SY_MAX_BLOCKS;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "smem attribute: %s", cudaGetErrorString(e)); return 4; }
    InboxMaps im;
    memset(&im, 0, sizeof im);
    for (int p = 0; p < cd.world; ++p)
      if (!make_map(&im.m[p], cd.heap[p] + inbox_off, (uint64_t)N, (uint64_t)cd.world * rpr, (uint64_t)N, kEpiChunk, BM)) return 3;
    kern<<<grid, kThreadsTN, smem, s>>>(ta, tb, im, cd, inbox_off, out_off, M, N, K, rpr);
    e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "launch: %s", cudaGetErrorString(e)); return 5; }
    g_launches.fetch_add(1);
    return 0;
  };
  switch (block_n) {
    case 64: return go(gemm_bf16_tn_rsag_kernel<64>, 64, Cfg<64>::kSmemBytes);
    case 128: return go(gemm_bf16_tn_rsag_kernel<128>, 128, Cfg<128>::kSmemBytes);
    case 256: return go(gemm_bf16_tn_rsag_kernel<256>, 256, Cfg<256>::kSmemBytes);
  }
  snprintf(g_err, sizeof g_err, "block_n must be 64, 128 or 256");
  return 1;
}

// C[M,N] = A[M,K] * B[K,N]; B row-major with N contiguous (MN-major operand, no transpose copy).  ldb % 8 == 0.
extern "C" int sy_gemm_bf16_nn(const void* A, const void* B, void* C, int M, int N, int K, int lda, int ldb, int ldc,
                               int block_n, int max_ctas, void* stream) {
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  if ((lda | ldb | ldc) & 7 || ((uintptr_t)A | (uintptr_t)B | (uintptr_t)C) & 15) {
    snprintf(g_err, sizeof g_err, "alignment: pointers must be 16B aligned and leading dimensions multiples of 8");
    return 1;
  }
  if (!load_encode()) { snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled unavailable (no driver?)"); return 6; }
  cudaStream_t s = (cudaStream_t)stream;
  if (block_n <= 0) block_n = N > 128 ? 256 : (N > 64 ? 128 : 64);
  switch (block_n) {
    case 64: return launch<64>(A, B, C, M, N, K, lda, ldb, ldc, nullptr, nullptr, max_ctas, s, true);
    case 128: return launch<128>(A, B, C, M, N, K, lda, ldb, ldc, nullptr, nullptr, max_ctas, s, true);
    case 256: return launch<256>(A, B, C, M, N, K, lda, ldb, ldc, nullptr, nullptr, max_ctas, s, true);
  }
  snprintf(g_err, sizeof g_err, "block_n must be 64, 128 or 256");
  return 1;
}

// Data gradient of a 1x1 / stride-2 convolution (the ResNet downsample branches): dX[Nb, 2P, 2Q, Cin] from dY[Nb*P*Q, Cout] and
// W[Cout, Cin] read in place (MN-major B).  One GEMM whose st.global epilogue scatters row (n, p, q) to pixel (2p, 2q) and writes the
// zeros of the three skipped pixels itself.  Cin % 8 == 0, pointers 16-byte aligned.
extern "C" int sy_gemm_bf16_nn_scatter2(const void* dY, const void* W, void* dX, int Nb, int P, int Q, int Cout, int Cin, int block_n,
                                        int max_ctas, void* stream) {
  const int M = Nb * P * Q, N = Cin, K = Cout;
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  if ((N | K) & 7 || ((uintptr_t)dY | (uintptr_t)W | (uintptr_t)dX) & 15) { snprintf(g_err, sizeof g_err, "scatter2: channels %% 8, 16B aligned pointers"); return 1; }
  if (!load_encode()) { snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled unavailable (no driver?)"); return 6; }
  if (block_n <= 0) block_n = N > 128 ? 256 : (N > 64 ? 128 : 64);
  auto go = [&](auto bn_tag) -> int {
    constexpr int BN = decltype(bn_tag)::value;
    using C = Cfg<BN>;
    CUtensorMap ta, tb, tc;
    if (!make_map(&ta, dY, K, M, K, BK, BM) || !make_map(&tb, W, N, K, N, 64, BK) || !make_map(&tc, dX, N, M, N, kEpiChunk, BM)) return 3;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);
    int grid = tiles < sms ? tiles : sms;
    if (max_ctas > 0 && grid > max_ctas) grid = max_ctas;
    auto kern = gemm_bf16_tn_kernel<BN, false, false, true, false, true>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes);
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "smem attribute: %s", cudaGetErrorString(e)); return 4; }
    ConvGeom g{P, Q, 1, 1, 0, 2, 0, 0};
    kern<<<grid, kThreadsTN, C::kSmemBytes, (cudaStream_t)stream>>>(ta, tb, tc, M, N, K, (const __nv_bfloat16*)nullptr, (float*)nullptr, g,
                                                                    (__nv_bfloat16*)dX, N, EpiAffine{});
    e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "launch: %s", cudaGetErrorString(e)); return 5; }
    g_launches.fetch_add(1);
    return 0;
  };
  switch (block_n) {
    case 64: return go(std::integral_constant<int, 64>{});
    case 128: return go(std::integral_constant<int, 128>{});
    case 256: return go(std::integral_constant<int, 256>{});
  }
  snprintf(g_err, sizeof g_err, "block_n must be 64, 128 or 256");
  return 1;
}

// out[j * ldo + i] (+)= sum_k A[k, i] * B[k, j]   (A: [K, I] row-major, B: [K, J] row-major; the wgrad shape).
// ws: float[I * J] and tickets: int[ceil(I/128) * ceil(J/block_n)], both zero on entry and zero again on exit.
// splits <= 0: chosen so that tiles * splits ~ number of SMs.
extern "C" int sy_gemm_bf16_nt_splitk(const void* A, const void* B, void* out, int I, int J, int K, int lda, int ldb, int ldo,
                                      float* ws, int* tickets, int accumulate, int block_n, int splits, void* stream) {
  if (I <= 0 || J <= 0 || K <= 0) return 0;
  if ((lda | ldb) & 7 || ((uintptr_t)A | (uintptr_t)B) & 15 || (ldo & 3) || ((uintptr_t)out & 7) || (I & 7)) {
    snprintf(g_err, sizeof g_err, "alignment: A/B 16B aligned, lda/ldb/I multiples of 8, out 8B aligned with ldo %% 4"); return 1;
  }
  if (!load_encode()) { snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled unavailable (no driver?)"); return 6; }
  if (block_n <= 0) block_n = J > 128 ? 256 : (J > 64 ? 128 : 64);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaStream_t s = (cudaStream_t)stream;
  auto go = [&](auto kern, int BN, int smem) -> int {
    CUtensorMap ta, tb;
    if (!make_map(&ta, A, I, K, lda, 64, BK) || !make_map(&tb, B, J, K, ldb, 64, BK)) return 3;
    const int tiles = ((I + BM - 1) / BM) * ((J + BN - 1) / BN), num_k = (K + BK - 1) / BK;
    int sp = splits;
    if (sp <= 0) { sp = sms / tiles; if (sp > num_k / 4) sp = num_k / 4; }
    if (sp < 1) sp = 1;
    if (sp > num_k) sp = num_k;
    if (sp > 1 && (!ws || !tickets)) { snprintf(g_err, sizeof g_err, "split-K needs a workspace"); return 2; }
    const long items = (long)tiles * sp;
    const int grid = (int)(items < sms ? items : sms);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "smem attribute: %s", cudaGetErrorString(e)); return 4; }
    kern<<<grid, kThreads, smem, s>>>(ta, tb, I, J, K, sp, ws, tickets, (__nv_bfloat16*)out, ldo, accumulate, ConvGeom{});
    e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "launch: %s", cudaGetErrorString(e)); return 5; }
    g_launches.fetch_add(1);
    return 0;
  };
  switch (block_n) {
    case 64: return go(gemm_bf16_nt_splitk_kernel<64, false>, 64, Cfg<64>::kSmemBytes);
    case 128: return go(gemm_bf16_nt_splitk_kernel<128, false>, 128, Cfg<128>::kSmemBytes);
    case 256: return go(gemm_bf16_nt_splitk_kernel<256, false>, 256, Cfg<256>::kSmemBytes);
  }
  snprintf(g_err, sizeof g_err, "block_n must be 64, 128 or 256");
  return 1;
}

// GEMM + all-reduce (K10).  `comm_view` = bytes of struct CommDev from sy_comm_device_view(); `out` is a
// symmetric fp32 [M, ldc] buffer at heap offset out_off, zeroed by the caller on every rank.
extern "C" int sy_gemm_bf16_tn_allreduce(const void* comm_view, size_t comm_view_bytes, const void* A, const void* B, size_t out_off,
                                         int M, int N, int K, int lda, int ldb, int ldc, int block_n, void* stream) {
  if (comm_view_bytes != sizeof(CommDev)) { snprintf(g_err, sizeof g_err, "communicator view size mismatch"); return 1; }
  if ((lda | ldb) & 7 || (ldc & 3) || (N & 3) || ((uintptr_t)A | (uintptr_t)B) & 15 || (out_off & 15)) {
    snprintf(g_err, sizeof g_err, "alignment: A/B 16B aligned, lda/ldb %% 8, N/ldc %% 4, out offset %% 16"); return 1;
  }
  if (!load_encode()) { snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled unavailable"); return 6; }
  CommDev cd; memcpy(&cd, comm_view, sizeof cd);
  if (block_n <= 0) block_n = N > 128 ? 256 : (N > 64 ? 128 : 64);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaStream_t s = (cudaStream_t)stream;
  auto go = [&](auto kern, int BN, int smem) -> int {
    CUtensorMap ta, tb;
    if (!make_map(&ta, A, K, M, lda, BK, BM) || !make_map(&tb, B, K, N, ldb, BK, BN)) return 3;
    const int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);
    int grid = tiles < sms ? tiles : sms;
    if (grid > SY_MAX_BLOCKS) grid = SY_MAX_BLOCKS;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "smem attribute: %s", cudaGetErrorString(e)); return 4; }
    kern<<<grid, kThreads, smem, s>>>(ta, tb, cd, out_off, ldc, M, N, K);
    e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(g_err, sizeof g_err, "launch: %s", cudaGetErrorString(e)); return 5; }
    g_launches.fetch_add(1);
    return 0;
  };
  switch (block_n) {
    case 64: return go(gemm_bf16_tn_allreduce_kernel<64>, 64, Cfg<64>::kSmemBytes);
    case 128: return go(gemm_bf16_tn_allreduce_kernel<128>, 128, Cfg<128>::kSmemBytes);
    case 256: return go(gemm_bf16_tn_allreduce_kernel<256>, 256, Cfg<256>::kSmemBytes);
  }
  snprintf(g_err, sizeof g_err, "block_n must be 64, 128 or 256");
  return 1;
}
