// Fused elementwise / normalisation kernels for the recipe workloads (sm_100a).
// All are HBM-bandwidth bound: 16-byte vector accesses, one pass over the data,
// statistics accumulated in fp32.  The reference has no kernels (SURVEY.md §2E); these serve the retargeted
// PyTorch-GPU recipe (/root/reference/recipes/PyTorch-GPU/config/jobs.yaml:1-8) and the HPCG retarget.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#define DEVI __device__ __forceinline__
struct alignas(16) V16 { uint32_t x, y, z, w; };

#include <atomic>
// counted across threads: autograd runs backward kernels from its own worker thread
static std::atomic<unsigned long long> g_launches{0};
extern "C" unsigned long long sy_ops_launch_count() { return g_launches.load(); }
#define COUNT_LAUNCH() do { g_launches.fetch_add(1, std::memory_order_relaxed); } while (0)
#define RET_LAST() do { cudaError_t e = cudaGetLastError(); return e == cudaSuccess ? 0 : (int)e; } while (0)

DEVI float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }
DEVI float bf_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
DEVI uint32_t pack_bf2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// ---------------------------------------------------------------------------
// uint8 NHWC image batch -> normalised bf16 NHWC (the step-input path: the
// staged uint8 batch is converted on the GPU, so H2D moves 1 byte per value)
// 16 input bytes (16 values) per thread -> 32 output bytes.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_u8_to_bf16_norm(const uint8_t* __restrict__ in, __nv_bfloat16* __restrict__ out, size_t n,
                  float m0, float m1, float m2, float s0, float s1, float s2) {
  const float mean[3] = {m0, m1, m2}, istd[3] = {s0, s1, s2};
  const size_t nv = n / 16;
  for (size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += (size_t)gridDim.x * blockDim.x) {
    const V16 raw = reinterpret_cast<const V16*>(in)[v];
    const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
    uint32_t o[8];
    int c = (int)((v * 16) % 3);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint32_t word = w[i / 2];
      const float a = (float)((word >> ((i % 2) * 16)) & 0xff);
      const float b = (float)((word >> ((i % 2) * 16 + 8)) & 0xff);
      const int c0 = c, c1 = c + 1 >= 3 ? c - 2 : c + 1;
      o[i] = pack_bf2((a * (1.f / 255.f) - mean[c0]) * istd[c0], (b * (1.f / 255.f) - mean[c1]) * istd[c1]);
      c = c1 + 1 >= 3 ? c1 - 2 : c1 + 1;
    }
    reinterpret_cast<V16*>(out)[2 * v] = V16{o[0], o[1], o[2], o[3]};
    reinterpret_cast<V16*>(out)[2 * v + 1] = V16{o[4], o[5], o[6], o[7]};
  }
  // tail (n % 16)
  for (size_t i = nv * 16 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % 3);
    out[i] = __float2bfloat16_rn(((float)in[i] * (1.f / 255.f) - mean[c]) * istd[c]);
  }
}

extern "C" int sy_ops_u8_to_bf16_norm(const void* in, void* out, size_t n, const float* mean3, const float* std3,
                                      void* stream) {
  size_t nv = n / 16 + 1;
  int blocks = (int)((nv + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  k_u8_to_bf16_norm<<<blocks, 256, 0, (cudaStream_t)stream>>>((const uint8_t*)in, (__nv_bfloat16*)out, n, mean3[0],
                                                              mean3[1], mean3[2], 1.f / std3[0], 1.f / std3[1], 1.f / std3[2]);
  COUNT_LAUNCH();
  RET_LAST();
}

// ===========================================================================
// Fused train-mode BatchNorm (+ residual add) (+ ReLU) on NHWC bf16 activations.
// x is the conv output viewed as [M, C] (M = N*H*W, C contiguous, C % 8 == 0,
// C/8 a power of two <= 256).  Thread t owns channel group t % (C/8) (8 channels,
// one 16-byte vector) and walks rows, so every access is a coalesced 16B vector
// and the per-channel parameters sit in registers.
//   fwd : stats (1 read)            -> apply (1-2 reads, 1 write)
//   bwd : reduce (3 reads)          -> apply (3 reads, 1-2 writes)
// versus separate BN / add / ReLU kernels this removes 2-4 full passes per layer.
// ===========================================================================
DEVI void unpack8(const V16& v, float* f) {
  f[0] = bf_lo(v.x); f[1] = bf_hi(v.x); f[2] = bf_lo(v.y); f[3] = bf_hi(v.y);
  f[4] = bf_lo(v.z); f[5] = bf_hi(v.z); f[6] = bf_lo(v.w); f[7] = bf_hi(v.w);
}
DEVI V16 pack8(const float* f) {
  return V16{pack_bf2(f[0], f[1]), pack_bf2(f[2], f[3]), pack_bf2(f[4], f[5]), pack_bf2(f[6], f[7])};
}
DEVI V16 ldg16(const void* p) {
  V16 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
DEVI void stg16(void* p, const V16& v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// block-level reduction of per-thread 8-channel partials, then one atomicAdd per channel
template <int NACC>
DEVI void block_reduce_atomic(float (&acc)[NACC][8], float* __restrict__ out, int C, int G) {
  __shared__ float sh[NACC][256][8];
#pragma unroll
  for (int a = 0; a < NACC; ++a)
#pragma unroll
    for (int i = 0; i < 8; ++i) sh[a][threadIdx.x][i] = acc[a][i];
  __syncthreads();
  // thread t < G*8 handles (channel group t/8, lane t%8)... use all 256 threads: (a, cg, i)
  const int items = NACC * G * 8;
  for (int it = threadIdx.x; it < items; it += blockDim.x) {
    const int a = it / (G * 8), cg = (it / 8) % G, i = it % 8;
    float s = 0.f;
    for (int t = cg; t < (int)blockDim.x; t += G) s += sh[a][t][i];
    atomicAdd(out + (size_t)a * C + cg * 8 + i, s);
  }
}

// Row loops are unrolled kU deep with every 16-byte load of a batch issued before the first use, so a
// thread keeps kU x (1-3) vectors in flight: HBM needs ~35 KB outstanding per SM (Little's law at
// 6.5 TB/s x ~800 ns) and 2 vectors per thread at ~50% occupancy is not enough.
constexpr int kU = 4;

__global__ void __launch_bounds__(256)
k_bn_stats(const __nv_bfloat16* __restrict__ x, float* __restrict__ sums, long M, int C) {
  const int G = C / 8, rpi = 256 / G, cg = threadIdx.x % G, rl = threadIdx.x / G;
  float acc[2][8] = {};
  const long stride = (long)gridDim.x * rpi;
  long r = (long)blockIdx.x * rpi + rl;
  auto body = [&](const V16& a) {
    float fa[8]; unpack8(a, fa);
#pragma unroll
    for (int i = 0; i < 8; ++i) { acc[0][i] += fa[i]; acc[1][i] = fmaf(fa[i], fa[i], acc[1][i]); }
  };
  for (; r + (2 * kU - 1) * stride < M; r += 2 * kU * stride) {
    V16 v[2 * kU];
#pragma unroll
    for (int u = 0; u < 2 * kU; ++u) v[u] = ldg16(x + (r + u * stride) * C + cg * 8);
#pragma unroll
    for (int u = 0; u < 2 * kU; ++u) body(v[u]);
  }
  for (; r < M; r += stride) body(ldg16(x + r * C + cg * 8));
  block_reduce_atomic<2>(acc, sums, C, G);
}

// out = act(gamma * (x - mean) * invstd + beta [+ res]); also finalises mean/invstd and running stats
__global__ void __launch_bounds__(256, 3)   // <= 85 registers: three resident blocks = 48 KB of loads in flight per SM
k_bn_apply_fwd(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ res,
               __nv_bfloat16* __restrict__ out, const float* __restrict__ sums,
               const __nv_bfloat16* __restrict__ gamma, const __nv_bfloat16* __restrict__ beta,
               float* __restrict__ running_mean, float* __restrict__ running_var,
               float* __restrict__ save_mean, float* __restrict__ save_invstd,
               long M, int C, float eps, float momentum, int relu, uint8_t* __restrict__ mask) {
  const int G = C / 8, rpi = 256 / G, cg = threadIdx.x % G, rl = threadIdx.x / G;
  float sc[8], sh[8];
  const float invM = 1.f / (float)M;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = cg * 8 + i;
    const float mean = sums[c] * invM;
    float var = sums[C + c] * invM - mean * mean;
    var = var < 0.f ? 0.f : var;
    const float istd = rsqrtf(var + eps);
    const float g = __bfloat162float(gamma[c]), b = __bfloat162float(beta[c]);
    sc[i] = g * istd; sh[i] = b - mean * g * istd;
    if (blockIdx.x == 0 && rl == 0) {
      save_mean[c] = mean; save_invstd[c] = istd;
      if (running_mean) {
        const float unb = M > 1 ? var * (float)M / (float)(M - 1) : var;
        running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * unb;
      }
    }
  }
  const long stride = (long)gridDim.x * rpi;
  // walk the rows from the END: the producer (conv / stats pass) touched the last rows most recently, so
  // whatever part of x still sits in the 126 MB L2 is consumed before it is evicted
  auto body = [&](long rr, const V16& vx, const V16& vr) {
    const size_t off = (size_t)rr * C + cg * 8;
    float f[8]; unpack8(vx, f);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = fmaf(f[i], sc[i], sh[i]);
    if (res) {
      float q[8]; unpack8(vr, q);
#pragma unroll
      for (int i = 0; i < 8; ++i) f[i] += q[i];
    }
    if (relu) {
      uint32_t bits = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) { bits |= (f[i] > 0.f ? 1u : 0u) << i; f[i] = fmaxf(f[i], 0.f); }
      // 1 bit per element for the backward pass: 16x less traffic than re-reading the activation
      if (mask) mask[(size_t)rr * G + cg] = (uint8_t)bits;
    }
    stg16(out + off, pack8(f));
  };
  long r = (long)blockIdx.x * rpi + rl;
  for (; r + (kU - 1) * stride < M; r += kU * stride) {
    V16 vx[kU], vr[kU];
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      const size_t off = (size_t)(M - 1 - (r + u * stride)) * C + cg * 8;
      vx[u] = ldg16(x + off);
      if (res) vr[u] = ldg16(res + off);
    }
#pragma unroll
    for (int u = 0; u < kU; ++u) body(M - 1 - (r + u * stride), vx[u], vr[u]);
  }
  for (; r < M; r += stride) {
    const size_t off = (size_t)(M - 1 - r) * C + cg * 8;
    V16 vr{}; if (res) vr = ldg16(res + off);
    body(M - 1 - r, ldg16(x + off), vr);
  }
}

DEVI void relu_gate(float* d, bool relu, bool has_mask, uint32_t bits, const V16& vo) {
  if (!relu) return;
  if (has_mask) {
#pragma unroll
    for (int i = 0; i < 8; ++i) d[i] = (bits >> i) & 1u ? d[i] : 0.f;
  } else {
    float o[8]; unpack8(vo, o);
#pragma unroll
    for (int i = 0; i < 8; ++i) d[i] = o[i] > 0.f ? d[i] : 0.f;
  }
}

// s1[c] = sum dz, s2[c] = sum dz * xhat, dz = relu ? dout * (out > 0) : dout
// kDual: the incoming gradient is the SUM of two tensors (a block output that feeds both the next block's first convolution
// and its residual connection): reading both here removes the separate add kernel autograd would run (read 2, write 1) and
// the re-read of its result.  The dual variant needs the saved ReLU bit mask (no `out` re-read), which keeps it at 111
// registers with the same 4-deep unroll (two resident blocks, like the single-gradient kernel).
template <bool kDual>
__global__ void __launch_bounds__(256)
k_bn_bwd_reduce(const __nv_bfloat16* __restrict__ dout, const __nv_bfloat16* __restrict__ dout2, const __nv_bfloat16* __restrict__ out,
                const __nv_bfloat16* __restrict__ x, const float* __restrict__ mean,
                const float* __restrict__ invstd, float* __restrict__ sums, long M, int C, int relu,
                const uint8_t* __restrict__ mask) {
  constexpr int U = kU;
  const int G = C / 8, rpi = 256 / G, cg = threadIdx.x % G, rl = threadIdx.x / G;
  float mu[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) mu[i] = mean[cg * 8 + i];
  float acc[2][8] = {};
  const long stride = (long)gridDim.x * rpi;
  const bool use_out = !kDual && relu && !mask;
  auto body = [&](const V16& vd, const V16& vd2, const V16& vx, uint32_t bits, const V16& vo) {
    float d[8], xv[8];
    unpack8(vd, d); unpack8(vx, xv);
    if constexpr (kDual) {
      float e[8]; unpack8(vd2, e);
#pragma unroll
      for (int i = 0; i < 8; ++i) d[i] += e[i];
    }
    relu_gate(d, relu, kDual || mask != nullptr, bits, vo);
#pragma unroll
    for (int i = 0; i < 8; ++i) { acc[0][i] += d[i]; acc[1][i] = fmaf(d[i], xv[i] - mu[i], acc[1][i]); }
  };
  long r = (long)blockIdx.x * rpi + rl;
  for (; r + (U - 1) * stride < M; r += U * stride) {
    V16 vd[U], vd2[U], vx[U], vo[U]; uint32_t mb[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long rr = r + u * stride;
      const size_t off = (size_t)rr * C + cg * 8;
      vd[u] = ldg16(dout + off); vx[u] = ldg16(x + off);
      if constexpr (kDual) vd2[u] = ldg16(dout2 + off);
      mb[u] = (relu && mask) ? mask[(size_t)rr * G + cg] : 0xffu;
      if (use_out) vo[u] = ldg16(out + off);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) body(vd[u], vd2[u], vx[u], mb[u], vo[u]);
  }
  for (; r < M; r += stride) {
    const size_t off = (size_t)r * C + cg * 8;
    V16 vo{}, v2{}; if (use_out) vo = ldg16(out + off);
    if constexpr (kDual) v2 = ldg16(dout2 + off);
    body(ldg16(dout + off), v2, ldg16(x + off), (relu && mask) ? mask[(size_t)r * G + cg] : 0xffu, vo);
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[1][i] *= invstd[cg * 8 + i];       // xhat = (x - mean) * invstd, factored out of the loop
  block_reduce_atomic<2>(acc, sums, C, G);
}

// dx = gamma*invstd*(dz - s1/M - xhat*s2/M); dres = dz; block 0 writes dgamma/dbeta (bf16)
template <bool kDual>
__global__ void __launch_bounds__(256)
k_bn_bwd_apply(const __nv_bfloat16* __restrict__ dout, const __nv_bfloat16* __restrict__ dout2, const __nv_bfloat16* __restrict__ out,
               const __nv_bfloat16* __restrict__ x, const float* __restrict__ mean,
               const float* __restrict__ invstd, const __nv_bfloat16* __restrict__ gamma,
               const float* __restrict__ sums, __nv_bfloat16* __restrict__ dx,
               __nv_bfloat16* __restrict__ dres, __nv_bfloat16* __restrict__ dgamma,
               __nv_bfloat16* __restrict__ dbeta, long M, int C, int relu, int accum, const uint8_t* __restrict__ mask) {
  constexpr int U = kU;
  const int G = C / 8, rpi = 256 / G, cg = threadIdx.x % G, rl = threadIdx.x / G;
  float k0[8], k1[8], k2[8];
  const float invM = 1.f / (float)M;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = cg * 8 + i;
    const float mu = mean[c], is = invstd[c];
    const float g = __bfloat162float(gamma[c]), s1 = sums[c], s2 = sums[C + c];
    // dx = g*is*dz + (-g*is*s2/M * is) * x + (-g*is*s1/M + g*is*s2/M * is * mu)
    k0[i] = g * is;
    k2[i] = -g * is * s2 * invM * is;
    k1[i] = -g * is * s1 * invM - k2[i] * mu;
    if (blockIdx.x == 0 && rl == 0) {
      // accum: add straight into the parameter's .grad view (no separate AccumulateGrad kernel)
      dgamma[c] = __float2bfloat16_rn(s2 + (accum ? __bfloat162float(dgamma[c]) : 0.f));
      dbeta[c] = __float2bfloat16_rn(s1 + (accum ? __bfloat162float(dbeta[c]) : 0.f));
    }
  }
  const long stride = (long)gridDim.x * rpi;
  const bool use_out = !kDual && relu && !mask;
  auto body = [&](long rr, const V16& vd, const V16& vd2, const V16& vx, uint32_t bits, const V16& vo) {
    const size_t off = (size_t)rr * C + cg * 8;
    float d[8], xv[8];
    unpack8(vd, d); unpack8(vx, xv);
    if constexpr (kDual) {
      float e[8]; unpack8(vd2, e);
#pragma unroll
      for (int i = 0; i < 8; ++i) d[i] += e[i];
    }
    relu_gate(d, relu, kDual || mask != nullptr, bits, vo);
    if (dres) stg16(dres + off, pack8(d));
    float g[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) g[i] = fmaf(d[i], k0[i], fmaf(xv[i], k2[i], k1[i]));
    stg16(dx + off, pack8(g));
  };
  // reversed row order: the reduce pass that ran just before ended on the last rows, so they are the ones in L2
  long r = (long)blockIdx.x * rpi + rl;
  for (; r + (U - 1) * stride < M; r += U * stride) {
    V16 vd[U], vd2[U], vx[U], vo[U]; uint32_t mb[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long rr = M - 1 - (r + u * stride);
      const size_t off = (size_t)rr * C + cg * 8;
      vd[u] = ldg16(dout + off); vx[u] = ldg16(x + off);
      if constexpr (kDual) vd2[u] = ldg16(dout2 + off);
      mb[u] = (relu && mask) ? mask[(size_t)rr * G + cg] : 0xffu;
      if (use_out) vo[u] = ldg16(out + off);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) body(M - 1 - (r + u * stride), vd[u], vd2[u], vx[u], mb[u], vo[u]);
  }
  for (; r < M; r += stride) {
    const long rr = M - 1 - r;
    const size_t off = (size_t)rr * C + cg * 8;
    V16 vo{}, v2{}; if (use_out) vo = ldg16(out + off);
    if constexpr (kDual) v2 = ldg16(dout2 + off);
    body(rr, ldg16(dout + off), v2, ldg16(x + off), (relu && mask) ? mask[(size_t)rr * G + cg] : 0xffu, vo);
  }
}

// blocks per SM: [0] stats (43 regs), [1] forward apply (88 regs), [2] backward reduce / apply (114 regs: 2 resident)
static int g_bn_bps[3] = {5, 3, 2};   // = resident blocks per SM of each kernel: exactly one wave
extern "C" void sy_ops_set_bn_blocks_per_sm(int n) { if (n > 0 && n <= 8) g_bn_bps[0] = g_bn_bps[1] = g_bn_bps[2] = n; }
extern "C" void sy_ops_set_bn_blocks_per_sm3(int stats, int fwd, int bwd) {
  if (stats > 0 && stats <= 8) g_bn_bps[0] = stats;
  if (fwd > 0 && fwd <= 8) g_bn_bps[1] = fwd;
  if (bwd > 0 && bwd <= 8) g_bn_bps[2] = bwd;
}
static inline int bn_grid(long M, int C, int which = 1) {
  const int g_bn_blocks_per_sm = g_bn_bps[which];
  const int rpi = 256 / (C / 8);
  long b = (M + rpi - 1) / rpi;
  b = (b + 3) / 4;                    // >= 4 rows per thread
  if (b > 148 * g_bn_blocks_per_sm) b = 148 * g_bn_blocks_per_sm;
  if (b < 1) b = 1;
  return (int)b;
}
static inline bool bn_shape_ok(int C) {
  if (C % 8) return false;
  int G = C / 8;
  return G >= 1 && G <= 256 && (G & (G - 1)) == 0;
}

// Callers that hand over scratch from a buffer they zeroed themselves (one memset per training step for ALL layers, see
// ops/fused.py zero pool) switch the per-call memsets off: ~85 memset nodes per ResNet-50 step otherwise.
static int g_ws_prezeroed = 0;
extern "C" void sy_ops_set_ws_prezeroed(int on) { g_ws_prezeroed = on ? 1 : 0; }

// ws: float[2*C] scratch (zeroed here unless sy_ops_set_ws_prezeroed(1)).  Returns 0 or a cuda error / -1 for bad shape.
extern "C" int sy_ops_bn_fwd(const void* x, const void* res, void* out, const void* gamma, const void* beta,
                             float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                             float* ws, long M, int C, float eps, float momentum, int relu, void* mask, void* stream) {
  if (!bn_shape_ok(C)) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  if (!g_ws_prezeroed) cudaMemsetAsync(ws, 0, sizeof(float) * 2 * C, s);
  const int g = bn_grid(M, C, 1);
  k_bn_stats<<<bn_grid(M, C, 0), 256, 0, s>>>((const __nv_bfloat16*)x, ws, M, C);
  COUNT_LAUNCH();
  k_bn_apply_fwd<<<g, 256, 0, s>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)res, (__nv_bfloat16*)out, ws,
                                   (const __nv_bfloat16*)gamma, (const __nv_bfloat16*)beta, running_mean, running_var,
                                   save_mean, save_invstd, M, C, eps, momentum, relu, (uint8_t*)mask);
  COUNT_LAUNCH();
  RET_LAST();
}

// variant used when the producing GEMM already accumulated the statistics in its epilogue
extern "C" int sy_ops_bn_apply_only(const void* x, const void* res, void* out, const void* gamma, const void* beta,
                                    float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                                    const float* sums, long M, int C, float eps, float momentum, int relu, void* mask, void* stream) {
  if (!bn_shape_ok(C)) return -1;
  const int g = bn_grid(M, C);
  k_bn_apply_fwd<<<g, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)res, (__nv_bfloat16*)out,
                                                      sums, (const __nv_bfloat16*)gamma, (const __nv_bfloat16*)beta, running_mean,
                                                      running_var, save_mean, save_invstd, M, C, eps, momentum, relu, (uint8_t*)mask);
  COUNT_LAUNCH();
  RET_LAST();
}

static int bn_bwd_launch(const void* dout, const void* dout2, const void* out, const void* x, const float* mean, const float* invstd,
                         const void* gamma, void* dx, void* dres, void* dgamma, void* dbeta, float* ws, long M, int C,
                         int relu, int accum, const void* mask, void* stream) {
  if (!bn_shape_ok(C)) return -1;
  if (dout2 && relu && !mask) return -2;          // the two-gradient variant gates with the saved bit mask only
  cudaStream_t s = (cudaStream_t)stream;
  if (!g_ws_prezeroed) cudaMemsetAsync(ws, 0, sizeof(float) * 2 * C, s);
  const int g = bn_grid(M, C, 2);
  auto D = [](const void* p) { return (const __nv_bfloat16*)p; };
  if (dout2) {
    k_bn_bwd_reduce<true><<<g, 256, 0, s>>>(D(dout), D(dout2), D(out), D(x), mean, invstd, ws, M, C, relu, (const uint8_t*)mask);
    COUNT_LAUNCH();
    k_bn_bwd_apply<true><<<g, 256, 0, s>>>(D(dout), D(dout2), D(out), D(x), mean, invstd, D(gamma), ws, (__nv_bfloat16*)dx, (__nv_bfloat16*)dres,
                                           (__nv_bfloat16*)dgamma, (__nv_bfloat16*)dbeta, M, C, relu, accum, (const uint8_t*)mask);
  } else {
    k_bn_bwd_reduce<false><<<g, 256, 0, s>>>(D(dout), nullptr, D(out), D(x), mean, invstd, ws, M, C, relu, (const uint8_t*)mask);
    COUNT_LAUNCH();
    k_bn_bwd_apply<false><<<g, 256, 0, s>>>(D(dout), nullptr, D(out), D(x), mean, invstd, D(gamma), ws, (__nv_bfloat16*)dx, (__nv_bfloat16*)dres,
                                            (__nv_bfloat16*)dgamma, (__nv_bfloat16*)dbeta, M, C, relu, accum, (const uint8_t*)mask);
  }
  COUNT_LAUNCH();
  RET_LAST();
}

extern "C" int sy_ops_bn_bwd(const void* dout, const void* out, const void* x, const float* mean, const float* invstd,
                             const void* gamma, void* dx, void* dres, void* dgamma, void* dbeta, float* ws, long M, int C,
                             int relu, int accum, const void* mask, void* stream) {
  return bn_bwd_launch(dout, nullptr, out, x, mean, invstd, gamma, dx, dres, dgamma, dbeta, ws, M, C, relu, accum, mask, stream);
}

// backward with the incoming gradient given as two tensors (dout + dout2 is formed in registers); needs `mask` when relu != 0
extern "C" int sy_ops_bn_bwd_dual(const void* dout, const void* dout2, const void* x, const float* mean, const float* invstd,
                                  const void* gamma, void* dx, void* dres, void* dgamma, void* dbeta, float* ws, long M, int C,
                                  int relu, int accum, const void* mask, void* stream) {
  return bn_bwd_launch(dout, dout2, nullptr, x, mean, invstd, gamma, dx, dres, dgamma, dbeta, ws, M, C, relu, accum, mask, stream);
}

// ===========================================================================
// 3x3 / stride 2 / pad 1 max-pool on NHWC bf16 with saved arg-max codes.
// fwd: one thread per (output pixel, 8-channel group): 9 x 16B loads, 16B store + 8 index bytes.
// bwd: one thread per (input pixel, 8-channel group): gathers from the <= 4 windows that cover
//      it (no atomics, every dx element written exactly once).
// ===========================================================================
// kIdx = false: inference variant without the arg-max codes (no index bytes written, no `code` registers)
template <bool kIdx>
__global__ void __launch_bounds__(256)
k_maxpool_fwd(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, uint8_t* __restrict__ idx,
              int N, int H, int W, int C, int OH, int OW) {
  const int G = C / 8;
  const long total = (long)N * OH * OW * G;
  for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
    const int g = (int)(t % G); long p = t / G;
    const int ox = (int)(p % OW); p /= OW;
    const int oy = (int)(p % OH); const int n = (int)(p / OH);
    float best[8]; uint32_t code[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { best[i] = -INFINITY; code[i] = 0; }
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int iy = 2 * oy - 1 + ky;
      if (iy < 0 || iy >= H) continue;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int ix = 2 * ox - 1 + kx;
        if (ix < 0 || ix >= W) continue;
        float f[8]; unpack8(ldg16(x + (((long)n * H + iy) * W + ix) * C + g * 8), f);
#pragma unroll
        for (int i = 0; i < 8; ++i) if (f[i] > best[i]) { best[i] = f[i]; if (kIdx) code[i] = ky * 3 + kx; }
      }
    }
    const long o = (((long)n * OH + oy) * OW + ox) * C + g * 8;
    stg16(y + o, pack8(best));
    if (!kIdx) continue;
    uint2 c2 = make_uint2(code[0] | (code[1] << 8) | (code[2] << 16) | (code[3] << 24), code[4] | (code[5] << 8) | (code[6] << 16) | (code[7] << 24));
    *reinterpret_cast<uint2*>(idx + o) = c2;
  }
}

__global__ void __launch_bounds__(256)
k_maxpool_bwd(const __nv_bfloat16* __restrict__ dy, const uint8_t* __restrict__ idx, __nv_bfloat16* __restrict__ dx,
              int N, int H, int W, int C, int OH, int OW) {
  const int G = C / 8;
  const long total = (long)N * H * W * G;
  for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
    const int g = (int)(t % G); long p = t / G;
    const int ix = (int)(p % W); p /= W;
    const int iy = (int)(p % H); const int n = (int)(p / H);
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    const int oy0 = iy / 2, oy1 = (iy + 1) / 2;     // windows with 2*oy-1 <= iy <= 2*oy+1
    const int ox0 = ix / 2, ox1 = (ix + 1) / 2;
    for (int oy = oy0; oy <= oy1; ++oy) {
      if (oy >= OH) continue;
      const int ky = iy - (2 * oy - 1);
      for (int ox = ox0; ox <= ox1; ++ox) {
        if (ox >= OW) continue;
        const int kx = ix - (2 * ox - 1);
        const uint32_t want = (uint32_t)(ky * 3 + kx);
        const long o = (((long)n * OH + oy) * OW + ox) * C + g * 8;
        const uint2 c2 = *reinterpret_cast<const uint2*>(idx + o);
        float d[8]; unpack8(ldg16(dy + o), d);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint32_t c = ((i < 4 ? c2.x : c2.y) >> (8 * (i & 3))) & 0xff;
          if (c == want) acc[i] += d[i];
        }
      }
    }
    stg16(dx + (((long)n * H + iy) * W + ix) * C + g * 8, pack8(acc));
  }
}

// Variant: one thread per 2x2 block of input pixels (and 8 channels).  The four pixels (2a..2a+1, 2b..2b+1) are covered by the same
// four pooling windows (oy in {a, a+1}, ox in {b, b+1}), so each window's gradient vector and arg-max codes are loaded once per
// thread instead of once per pixel (96 B of loads per 64 B stored instead of 216 B) and every thread has four independent 16-byte
// stores in flight.  ncu (profiles/step_breakdown.md) has the per-pixel kernel at 494 us for the 411 MB stem gradient, 5x the HBM time.
// Default since round 2 for even H and W (bit-compared against the per-pixel kernel on hardware, tests/test_zz_gpu_bn_dual.py; step 20.81 ->
// 20.57 ms in the same call, gpurun_out/r2_bench_pool2.json); SHIPYARD_MAXPOOL_BWD2=0 selects the per-pixel kernel.
__global__ void __launch_bounds__(256)
k_maxpool_bwd2(const __nv_bfloat16* __restrict__ dy, const uint8_t* __restrict__ idx, __nv_bfloat16* __restrict__ dx,
               int N, int H, int W, int C, int OH, int OW) {
  const int G = C / 8, H2 = H / 2, W2 = W / 2;
  const long total = (long)N * H2 * W2 * G;
  for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
    const int g = (int)(t % G); long p = t / G;
    const int b = (int)(p % W2); p /= W2;
    const int a = (int)(p % H2); const int n = (int)(p / H2);
    float acc[2][2][8];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[i][j][c] = 0.f;
#pragma unroll
    for (int wy = 0; wy < 2; ++wy) {
      const int oy = a + wy;
      if (oy >= OH) continue;
#pragma unroll
      for (int wx = 0; wx < 2; ++wx) {
        const int ox = b + wx;
        if (ox >= OW) continue;
        const long o = (((long)n * OH + oy) * OW + ox) * C + g * 8;
        const uint2 c2 = *reinterpret_cast<const uint2*>(idx + o);
        float d[8]; unpack8(ldg16(dy + o), d);
        // window (oy, ox) covers input rows 2*oy-1 .. 2*oy+1: of this block's rows 2a, 2a+1 that is ky = 1, 2 (wy = 0) or ky = -, 0 (wy = 1)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int ky = 2 * a + i - (2 * oy - 1);
          if (ky < 0 || ky > 2) continue;
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const int kx = 2 * b + j - (2 * ox - 1);
            if (kx < 0 || kx > 2) continue;
            const uint32_t want = (uint32_t)(ky * 3 + kx);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const uint32_t code = ((c < 4 ? c2.x : c2.y) >> (8 * (c & 3))) & 0xff;
              if (code == want) acc[i][j][c] += d[c];
            }
          }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j)
        stg16(dx + (((long)n * H + 2 * a + i) * W + 2 * b + j) * C + g * 8, pack8(acc[i][j]));
  }
}

// idx == NULL: inference (no arg-max codes, nothing for a backward pass)
extern "C" int sy_ops_maxpool3x3s2_fwd(const void* x, void* y, void* idx, int N, int H, int W, int C, void* stream) {
  if (C % 8) return -1;
  const int OH = (H + 2 - 3) / 2 + 1, OW = (W + 2 - 3) / 2 + 1;
  long total = (long)N * OH * OW * (C / 8);
  int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  if (idx)
    k_maxpool_fwd<true><<<blocks, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)y, (uint8_t*)idx, N, H, W, C, OH, OW);
  else
    k_maxpool_fwd<false><<<blocks, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)y, nullptr, N, H, W, C, OH, OW);
  COUNT_LAUNCH();
  RET_LAST();
}
extern "C" int sy_ops_maxpool3x3s2_bwd(const void* dy, const void* idx, void* dx, int N, int H, int W, int C, void* stream) {
  if (C % 8) return -1;
  const int OH = (H + 2 - 3) / 2 + 1, OW = (W + 2 - 3) / 2 + 1;
  static int bwd2 = -1;
  if (bwd2 < 0) { const char* e = getenv("SHIPYARD_MAXPOOL_BWD2"); bwd2 = (e && e[0] == '0') ? 0 : 1; }
  if (bwd2 && H % 2 == 0 && W % 2 == 0) {
    const long total2 = (long)N * (H / 2) * (W / 2) * (C / 8);
    const int blocks2 = (int)((total2 + 255) / 256 < 148 * 16 ? (total2 + 255) / 256 : 148 * 16);
    k_maxpool_bwd2<<<blocks2, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)dy, (const uint8_t*)idx, (__nv_bfloat16*)dx, N, H, W, C, OH, OW);
    COUNT_LAUNCH();
    RET_LAST();
  }
  long total = (long)N * H * W * (C / 8);
  int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  k_maxpool_bwd<<<blocks, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)dy, (const uint8_t*)idx, (__nv_bfloat16*)dx, N, H, W, C, OH, OW);
  COUNT_LAUNCH();
  RET_LAST();
}

// ===========================================================================
// Inference BatchNorm.  The fold turns every BN layer of a model into a per-channel affine map in ONE launch (one block per
// layer), reading the parameters and running statistics where they live, so a captured inference graph always applies the
// current values:  scale = gamma * rsqrt(running_var + eps),  shift = beta - running_mean * scale.
// bn_infer_apply is the same map as a stand-alone pass for layers whose convolution has no fused epilogue:
//   out = act(x * scale + shift (+ residual))  on NHWC bf16 [M, C], C % 8 == 0, 16-byte vectors.
// ===========================================================================
struct BnFoldEntry {                  // 64 bytes, laid out by ops/fused.py (eight 64-bit words)
  const __nv_bfloat16* gamma;
  const __nv_bfloat16* beta;
  const float* running_mean;
  const float* running_var;
  float* scale_out;
  float* shift_out;
  long long C;
  float eps;
  float pad_;
};

__global__ void __launch_bounds__(256)
k_bn_fold(const BnFoldEntry* __restrict__ table) {
  const BnFoldEntry e = table[blockIdx.x];
  for (int c = threadIdx.x; c < (int)e.C; c += blockDim.x) {
    const float sc = __bfloat162float(e.gamma[c]) * rsqrtf(e.running_var[c] + e.eps);
    e.scale_out[c] = sc;
    e.shift_out[c] = __bfloat162float(e.beta[c]) - e.running_mean[c] * sc;
  }
}

extern "C" int sy_ops_bn_fold(const void* table, int n_layers, void* stream) {
  if (n_layers <= 0) return 0;
  k_bn_fold<<<n_layers, 256, 0, (cudaStream_t)stream>>>((const BnFoldEntry*)table);
  COUNT_LAUNCH();
  RET_LAST();
}

__global__ void __launch_bounds__(256)
k_bn_infer_apply(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ res, __nv_bfloat16* out,
                 const float* __restrict__ scale, const float* __restrict__ shift, long nvec, int G, int relu) {
  for (long v = (long)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += (long)gridDim.x * blockDim.x) {
    const int cg = (int)(v % G);
    const V16 vx = ldg16(x + v * 8);
    V16 vr{};
    if (res) vr = ldg16(res + v * 8);
    const float4 s0 = __ldg(reinterpret_cast<const float4*>(scale) + 2 * cg), s1 = __ldg(reinterpret_cast<const float4*>(scale) + 2 * cg + 1);
    const float4 t0 = __ldg(reinterpret_cast<const float4*>(shift) + 2 * cg), t1 = __ldg(reinterpret_cast<const float4*>(shift) + 2 * cg + 1);
    const float s[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
    const float t[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
    float f[8], r[8];
    unpack8(vx, f); unpack8(vr, r);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      f[i] = fmaf(f[i], s[i], t[i]) + r[i];
      if (relu) f[i] = fmaxf(f[i], 0.f);
    }
    stg16(out + v * 8, pack8(f));
  }
}

// x, res (optional), out: [M, C] bf16, 16-byte aligned; scale / shift: fp32[C], 16-byte aligned.  out may be x (in place).
extern "C" int sy_ops_bn_infer_apply(const void* x, const void* res, void* out, const float* scale, const float* shift, long M, int C,
                                     int relu, void* stream) {
  if (C % 8 || M < 0 || (((uintptr_t)x | (uintptr_t)res | (uintptr_t)out | (uintptr_t)scale | (uintptr_t)shift) & 15)) return -1;
  const long nvec = M * (C / 8);
  if (nvec == 0) return 0;
  long blocks = (nvec + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  k_bn_infer_apply<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)res, (__nv_bfloat16*)out,
                                                                  scale, shift, nvec, C / 8, relu);
  COUNT_LAUNCH();
  RET_LAST();
}

// ===========================================================================
// Stem input transform: uint8 NHWC [N,H,W,3] -> normalised bf16 space-to-depth [N, H/2+3, W/2+3, 16]
// with a zero border (2 before, 1 after) so that the 7x7/stride-2/pad-3 stem convolution becomes a
// dense 4x4/stride-1/pad-0 convolution over 16 channels (12 used): channel (p*2+q)*3+c of cell (Y,X)
// holds pixel (2(Y-2)+p, 2(X-2)+q, c).  One thread writes one 32-byte cell.
// ===========================================================================
__global__ void __launch_bounds__(256)
k_u8_to_s2d(const uint8_t* __restrict__ in, __nv_bfloat16* __restrict__ out, int N, int H, int W,
            float m0, float m1, float m2, float s0, float s1, float s2) {
  const int OH = H / 2 + 3, OW = W / 2 + 3;
  const float mean[3] = {m0, m1, m2}, istd[3] = {s0, s1, s2};
  const long total = (long)N * OH * OW;
  for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
    const int X = (int)(t % OW); long p = t / OW;
    const int Y = (int)(p % OH); const int n = (int)(p / OH);
    float f[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) f[i] = 0.f;
    const int y0 = 2 * (Y - 2), x0 = 2 * (X - 2);
    if (Y >= 2 && X >= 2 && y0 + 1 < H && x0 + 1 < W) {
#pragma unroll
      for (int pp = 0; pp < 2; ++pp) {
        const uint8_t* src = in + (((long)n * H + y0 + pp) * W + x0) * 3;   // 6 consecutive bytes: (q=0,c=0..2),(q=1,c=0..2)
#pragma unroll
        for (int j = 0; j < 6; ++j) f[pp * 6 + j] = ((float)src[j] * (1.f / 255.f) - mean[j % 3]) * istd[j % 3];
      }
    }
    stg16(out + t * 16, pack8(f));
    stg16(out + t * 16 + 8, pack8(f + 8));
  }
}

extern "C" int sy_ops_u8_to_s2d_norm(const void* in, void* out, int N, int H, int W, const float* mean3, const float* std3, void* stream) {
  if ((H | W) & 1) return -1;
  long total = (long)N * (H / 2 + 3) * (W / 2 + 3);
  int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  k_u8_to_s2d<<<blocks, 256, 0, (cudaStream_t)stream>>>((const uint8_t*)in, (__nv_bfloat16*)out, N, H, W, mean3[0], mean3[1], mean3[2],
                                                       1.f / std3[0], 1.f / std3[1], 1.f / std3[2]);
  COUNT_LAUNCH();
  RET_LAST();
}

// ===========================================================================
// HPCG retarget kernels (fp64, 27-point stencil, matrix-free: diagonal 26, off-diagonals -1 for every
// neighbour inside the global domain).  The local grid is nx*ny*nz with a 1-D decomposition along z;
// the z-neighbour planes arrive in `lo` / `hi` ghost buffers written by the neighbours' fused halo push.
// ===========================================================================
DEVI double stencil_nbr_sum(const double* __restrict__ x, const double* __restrict__ lo, const double* __restrict__ hi,
                            int ix, int iy, int iz, int nx, int ny, int nz, int* count) {
  double s = 0.0; int c = 0;
#pragma unroll
  for (int dz = -1; dz <= 1; ++dz) {
    const int z = iz + dz;
    const double* plane;
    if (z < 0) { if (!lo) continue; plane = lo; }
    else if (z >= nz) { if (!hi) continue; plane = hi; }
    else plane = x + (size_t)z * nx * ny;
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy) {
      const int y = iy + dy;
      if (y < 0 || y >= ny) continue;
#pragma unroll
      for (int dx = -1; dx <= 1; ++dx) {
        const int xx = ix + dx;
        if (xx < 0 || xx >= nx || (dx == 0 && dy == 0 && dz == 0)) continue;
        s += plane[(size_t)y * nx + xx]; ++c;
      }
    }
  }
  if (count) *count = c;
  return s;
}

__global__ void __launch_bounds__(256)
k_hpcg_spmv(const double* __restrict__ x, const double* __restrict__ lo, const double* __restrict__ hi, double* __restrict__ y,
            int nx, int ny, int nz) {
  const size_t n = (size_t)nx * ny * nz;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int ix = (int)(i % nx), iy = (int)((i / nx) % ny), iz = (int)(i / ((size_t)nx * ny));
    y[i] = 26.0 * x[i] - stencil_nbr_sum(x, lo, hi, ix, iy, iz, nx, ny, nz, nullptr);
  }
}

// one colour of the 8-colour Gauss-Seidel sweep: x_i = (r_i + sum of neighbours) / 26
__global__ void __launch_bounds__(256)
k_hpcg_symgs_color(const double* __restrict__ r, double* __restrict__ x, const double* __restrict__ lo, const double* __restrict__ hi,
                   int nx, int ny, int nz, int color, int zoff) {
  const int cx = color & 1, cy = (color >> 1) & 1, cz = (color >> 2) & 1;
  const int hx = (nx - cx + 1) / 2, hy = (ny - cy + 1) / 2;
  const int z0 = ((cz - zoff) % 2 + 2) % 2;             // first local z with global parity cz
  const int hz = (nz - z0 + 1) / 2;
  const size_t n = (size_t)hx * hy * hz;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (size_t)gridDim.x * blockDim.x) {
    const int ix = 2 * (int)(t % hx) + cx, iy = 2 * (int)((t / hx) % hy) + cy, iz = 2 * (int)(t / ((size_t)hx * hy)) + z0;
    const size_t i = ((size_t)iz * ny + iy) * nx + ix;
    x[i] = (r[i] + stencil_nbr_sum(x, lo, hi, ix, iy, iz, nx, ny, nz, nullptr)) * (1.0 / 26.0);
  }
}

// b = A * ones  (26 - number of in-domain neighbours); gz0 / gnz give this rank's place in the global z range
__global__ void k_hpcg_rhs(double* __restrict__ b, int nx, int ny, int nz, int gz0, int gnz) {
  const size_t n = (size_t)nx * ny * nz;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int ix = (int)(i % nx), iy = (int)((i / nx) % ny), iz = (int)(i / ((size_t)nx * ny)) + gz0;
    const int cx = 1 + (ix > 0) + (ix < nx - 1), cy = 1 + (iy > 0) + (iy < ny - 1), cz = 1 + (iz > 0) + (iz < gnz - 1);
    b[i] = 26.0 - (double)(cx * cy * cz - 1);
  }
}

// coarse residual: rc[c] = rf[f] - Axf[f] at f = (2x, 2y, 2z)
__global__ void k_hpcg_restrict(const double* __restrict__ rf, const double* __restrict__ axf, double* __restrict__ rc, int nxc, int nyc, int nzc) {
  const size_t n = (size_t)nxc * nyc * nzc;
  const int nxf = 2 * nxc, nyf = 2 * nyc;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int ix = (int)(i % nxc), iy = (int)((i / nxc) % nyc), iz = (int)(i / ((size_t)nxc * nyc));
    const size_t f = ((size_t)(2 * iz) * nyf + 2 * iy) * nxf + 2 * ix;
    rc[i] = rf[f] - axf[f];
  }
}
__global__ void k_hpcg_prolong(double* __restrict__ xf, const double* __restrict__ xc, int nxc, int nyc, int nzc) {
  const size_t n = (size_t)nxc * nyc * nzc;
  const int nxf = 2 * nxc, nyf = 2 * nyc;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int ix = (int)(i % nxc), iy = (int)((i / nxc) % nyc), iz = (int)(i / ((size_t)nxc * nyc));
    xf[((size_t)(2 * iz) * nyf + 2 * iy) * nxf + 2 * ix] += xc[i];
  }
}

static inline int hpcg_grid(size_t n) { size_t b = (n + 255) / 256; return (int)(b < 148 * 8 ? (b ? b : 1) : 148 * 8); }
extern "C" int sy_hpcg_spmv(const void* x, const void* lo, const void* hi, void* y, int nx, int ny, int nz, void* stream) {
  k_hpcg_spmv<<<hpcg_grid((size_t)nx * ny * nz), 256, 0, (cudaStream_t)stream>>>((const double*)x, (const double*)lo, (const double*)hi, (double*)y, nx, ny, nz);
  COUNT_LAUNCH(); RET_LAST();
}
// one symmetric sweep: colours 0..7 then 7..0
extern "C" int sy_hpcg_symgs(const void* r, void* x, const void* lo, const void* hi, int nx, int ny, int nz, int zoff, void* stream) {
  const int g = hpcg_grid((size_t)nx * ny * nz / 8 + 1);
  for (int pass = 0; pass < 2; ++pass)
    for (int k = 0; k < 8; ++k) {
      const int color = pass == 0 ? k : 7 - k;
      k_hpcg_symgs_color<<<g, 256, 0, (cudaStream_t)stream>>>((const double*)r, (double*)x, (const double*)lo, (const double*)hi, nx, ny, nz, color, zoff);
      COUNT_LAUNCH();
    }
  RET_LAST();
}
extern "C" int sy_hpcg_rhs(void* b, int nx, int ny, int nz, int gz0, int gnz, void* stream) {
  k_hpcg_rhs<<<hpcg_grid((size_t)nx * ny * nz), 256, 0, (cudaStream_t)stream>>>((double*)b, nx, ny, nz, gz0, gnz);
  COUNT_LAUNCH(); RET_LAST();
}
extern "C" int sy_hpcg_restrict(const void* rf, const void* axf, void* rc, int nxc, int nyc, int nzc, void* stream) {
  k_hpcg_restrict<<<hpcg_grid((size_t)nxc * nyc * nzc), 256, 0, (cudaStream_t)stream>>>((const double*)rf, (const double*)axf, (double*)rc, nxc, nyc, nzc);
  COUNT_LAUNCH(); RET_LAST();
}
extern "C" int sy_hpcg_prolong(void* xf, const void* xc, int nxc, int nyc, int nzc, void* stream) {
  k_hpcg_prolong<<<hpcg_grid((size_t)nxc * nyc * nzc), 256, 0, (cudaStream_t)stream>>>((double*)xf, (const double*)xc, nxc, nyc, nzc);
  COUNT_LAUNCH(); RET_LAST();
}
