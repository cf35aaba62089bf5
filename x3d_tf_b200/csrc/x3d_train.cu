// Training-step kernels (BASELINE.json configs[4]: X3D-M training step), fp32, channels-last.
// First correct versions: every operation the Keras train_step of the reference performs around
// the convolutions (train.py:85-152 -> model.py with training=True) as hand-written CUDA --
// batch-statistics BatchNorm forward/backward, backward-data / backward-filter of the pointwise,
// channelwise and stem convolutions, SE / swish / ReLU / dropout / pooling backward, softmax
// cross-entropy, SGD-Nesterov with L2.  They are coalesced and grid-sized for 148 SMs but not yet
// tuned (DESIGN.md section 9 lists what the tuned versions will fuse).
//
// Reductions over the row dimension accumulate per-thread in fp32 over short row runs, then in
// fp64 through atomicAdd(double): the fp64 sum of <= 2^24 fp32 partials is exact to ~1e-13
// relative, so results do not depend on the arrival order after rounding to fp32.
#include "common.cuh"

namespace x3d {
namespace train {

static inline cudaStream_t S(void* s) { return static_cast<cudaStream_t>(s); }
constexpr int kRowsPerBlock = 256;

// ---------------------------------------------------------------- per-channel row reductions
// mode 0: out[0][c] += sum a,        out[1][c] += sum a*a            (BN statistics)
// mode 1: out[0][c] += sum g,        out[1][c] += sum g * xhat       (BN backward; g = dy masked
//         by relu_out > 0 when relu_out != nullptr; xhat = (x - mean) * rstd)
// mode 2: out[0][c] += sum a                                          (bias gradients)
// Rows are split in segments of `seg_rows` (one output row pair per segment: per-clip sums).
__global__ void __launch_bounds__(256)
colreduce_kernel(const float* __restrict__ a, const float* __restrict__ x, const float* __restrict__ mean,
                 const float* __restrict__ rstd, const float* __restrict__ relu_out, long M, int C,
                 long seg_rows, double* __restrict__ out, int mode) {
  const int cx = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ry = threadIdx.x >> 5;                       // 8 row lanes
  const long seg = blockIdx.z;
  const long r0 = seg * seg_rows + (long)blockIdx.y * kRowsPerBlock;
  long r1 = r0 + kRowsPerBlock;
  const long seg_end = (seg + 1) * seg_rows < M ? (seg + 1) * seg_rows : M;
  if (r1 > seg_end) r1 = seg_end;
  float s0 = 0.f, s1 = 0.f;
  if (cx < C) {
    const float mu = (mode == 1) ? mean[cx] : 0.f, rs = (mode == 1) ? rstd[cx] : 0.f;
    for (long r = r0 + ry; r < r1; r += 8) {
      const float v = a[r * C + cx];
      if (mode == 0) { s0 += v; s1 = fmaf(v, v, s1); }
      else if (mode == 1) {
        const float g = (relu_out == nullptr || relu_out[r * C + cx] > 0.f) ? v : 0.f;
        s0 += g; s1 = fmaf(g, (x[r * C + cx] - mu) * rs, s1);
      } else s0 += v;
    }
  }
  __shared__ float sh0[8][33], sh1[8][33];
  sh0[ry][threadIdx.x & 31] = s0; sh1[ry][threadIdx.x & 31] = s1;
  __syncthreads();
  if (ry == 0 && cx < C) {
    double t0 = 0.0, t1 = 0.0;
    for (int i = 0; i < 8; ++i) { t0 += sh0[i][threadIdx.x]; t1 += sh1[i][threadIdx.x]; }
    atomicAdd(out + (seg * 2) * C + cx, t0);
    if (mode != 2) atomicAdd(out + (seg * 2 + 1) * C + cx, t1);
  }
}

// The same sums for ONE segment (BN statistics / BN backward over the whole batch) with 128-bit loads:
// thread i walks the [M, C/4] float4 matrix at i, i + stride4, ... with stride4 a multiple of C/4, so it
// stays on the same four channels and keeps 8 running sums in registers, four rows in flight per stream.
// The block's sums meet in shared memory and are added per channel in thread order in fp64 (the same
// result for the same launch geometry), then one fp64 atomic per channel and block goes to `out` -- the
// scalar kernel above reached ~25 % of HBM
// (one 4-byte load per thread and row, 208 launches = 9.9 ms of the X3D-M step).
__global__ void __launch_bounds__(256)
colreduce_vec_kernel(const float* __restrict__ a, const float* __restrict__ x, const float* __restrict__ mean,
                     const float* __restrict__ rstd, const float* __restrict__ relu_out, long total4, int C4,
                     long stride4, double* __restrict__ out, int mode) {
  __shared__ float part[8][256];                          // [sum j of 4 channels x 2][thread]
  const int C = C4 << 2;
  const long i0 = (long)blockIdx.x * blockDim.x + threadIdx.x;
  float s0[4] = {0.f, 0.f, 0.f, 0.f}, s1[4] = {0.f, 0.f, 0.f, 0.f};
  if (i0 < total4 && i0 < stride4) {
    const int c = (int)(i0 % C4) << 2;
    float mu[4] = {0.f, 0.f, 0.f, 0.f}, rs[4] = {0.f, 0.f, 0.f, 0.f};
    if (mode == 1) {
#pragma unroll
      for (int j = 0; j < 4; ++j) { mu[j] = mean[c + j]; rs[j] = rstd[c + j]; }
    }
    const float4* a4 = reinterpret_cast<const float4*>(a);
    const float4* x4 = reinterpret_cast<const float4*>(x);
    const float4* r4 = reinterpret_cast<const float4*>(relu_out);
    auto add = [&](const float4& av, const float4& xv, const float4& rv) {
      const float v[4] = {av.x, av.y, av.z, av.w};
      const float xx[4] = {xv.x, xv.y, xv.z, xv.w};
      const float rr[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (mode == 0) { s0[j] += v[j]; s1[j] = fmaf(v[j], v[j], s1[j]); }
        else if (mode == 1) {
          const float g = rr[j] > 0.f ? v[j] : 0.f;
          s0[j] += g; s1[j] = fmaf(g, (xx[j] - mu[j]) * rs[j], s1[j]);
        } else s0[j] += v[j];
      }
    };
    const float4 one = make_float4(1.f, 1.f, 1.f, 1.f), zero = make_float4(0.f, 0.f, 0.f, 0.f);
    long i = i0;
    for (; i + 3 * stride4 < total4; i += 4 * stride4) {
      float4 av[4], xv[4], rv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        av[u] = __ldg(a4 + i + u * stride4);
        xv[u] = mode == 1 ? __ldg(x4 + i + u * stride4) : zero;
        rv[u] = (mode == 1 && r4 != nullptr) ? __ldg(r4 + i + u * stride4) : one;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) add(av[u], xv[u], rv[u]);
    }
    for (; i < total4; i += stride4)
      add(__ldg(a4 + i), mode == 1 ? __ldg(x4 + i) : zero, (mode == 1 && r4 != nullptr) ? __ldg(r4 + i) : one);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) { part[j][threadIdx.x] = s0[j]; part[4 + j][threadIdx.x] = s1[j]; }
  __syncthreads();
  // thread t of this block works on channel group (first + t) mod C4
  const int first = (int)(((long)blockIdx.x * blockDim.x) % C4);
  for (int i = threadIdx.x; i < (mode != 2 ? 2 : 1) * C; i += blockDim.x) {
    const int which = i >= C ? 1 : 0, c = i - which * C, g = c >> 2, j = c & 3;
    double t = 0.0;
    for (int th = (g - first + C4) % C4; th < 256; th += C4) t += (double)part[which * 4 + j][th];
    atomicAdd(out + i, t);
  }
}

// BN statistics from the fp64 sums: mean, biased variance (TF BatchNormalization, model.py:89,196,
// 254,268,300,368 in training mode), rstd = 1/sqrt(var+eps); moving stats updated in place with
// momentum m: moving = m*moving + (1-m)*batch (configs/default.py:43).
__global__ void bn_finalize_kernel(const double* __restrict__ sums, long M, int C, float eps, float momentum,
                                   float* __restrict__ mean, float* __restrict__ var, float* __restrict__ rstd,
                                   float* __restrict__ mov_mean, float* __restrict__ mov_var) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double mu = sums[c] / (double)M;
  double v = sums[C + c] / (double)M - mu * mu;
  if (v < 0.0) v = 0.0;
  mean[c] = (float)mu; var[c] = (float)v; rstd[c] = (float)(1.0 / sqrt(v + (double)eps));
  if (mov_mean) mov_mean[c] = momentum * mov_mean[c] + (1.f - momentum) * (float)mu;
  if (mov_var) mov_var[c] = momentum * mov_var[c] + (1.f - momentum) * (float)v;
}

// y = (x - mean) * rstd * gamma + beta  (+ ReLU).  128-bit accesses; the per-channel scale/shift of
// a thread's 4 channels are combined once (the grid stride is a multiple of C/4 float4 columns, so a
// thread stays on the same channels) -- no 64-bit modulo and 4 table reads per element.
__global__ void __launch_bounds__(256)
bn_apply_kernel(const float* __restrict__ x, const float* __restrict__ mean, const float* __restrict__ rstd,
                const float* __restrict__ gamma, const float* __restrict__ beta, float* __restrict__ y,
                long total4, int C4, long stride4, int relu) {
  const long i0 = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i0 >= total4 || i0 >= stride4) return;
  const int c = (int)(i0 % C4) << 2;
  float sc[4], sh[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    sc[j] = rstd[c + j] * gamma[c + j];
    sh[j] = beta[c + j] - mean[c + j] * sc[j];
  }
  const float4* x4 = reinterpret_cast<const float4*>(x);
  float4* y4 = reinterpret_cast<float4*>(y);
  for (long i = i0; i < total4; i += stride4) {
    const float4 v = __ldg(x4 + i);
    float4 r = make_float4(fmaf(v.x, sc[0], sh[0]), fmaf(v.y, sc[1], sh[1]), fmaf(v.z, sc[2], sh[2]), fmaf(v.w, sc[3], sh[3]));
    if (relu) r = make_float4(fmaxf(r.x, 0.f), fmaxf(r.y, 0.f), fmaxf(r.z, 0.f), fmaxf(r.w, 0.f));
    y4[i] = r;
  }
}

// dx = gamma * rstd * (g - sum_g/M - xhat * sum_gx/M),  g = dy masked by relu_out > 0; same layout.
__global__ void __launch_bounds__(256)
bn_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ relu_out,
                    const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ gamma,
                    const double* __restrict__ sums, float* __restrict__ dx, long total4, int C4, long stride4, long M) {
  const long i0 = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i0 >= total4 || i0 >= stride4) return;
  const int C = C4 << 2, c = (int)(i0 % C4) << 2;
  const double invM = 1.0 / (double)M;
  float mu[4], rs[4], k[4], sg[4], sgx[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    mu[j] = mean[c + j]; rs[j] = rstd[c + j]; k[j] = gamma[c + j] * rs[j];
    sg[j] = (float)(sums[c + j] * invM); sgx[j] = (float)(sums[C + c + j] * invM);
  }
  const float4* dy4 = reinterpret_cast<const float4*>(dy);
  const float4* x4 = reinterpret_cast<const float4*>(x);
  const float4* r4 = reinterpret_cast<const float4*>(relu_out);
  float4* dx4 = reinterpret_cast<float4*>(dx);
  for (long i = i0; i < total4; i += stride4) {
    const float4 gv = __ldg(dy4 + i), xv = __ldg(x4 + i);
    float g[4] = {gv.x, gv.y, gv.z, gv.w};
    const float xx[4] = {xv.x, xv.y, xv.z, xv.w};
    if (r4 != nullptr) {
      const float4 rv = __ldg(r4 + i);
      const float rr[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) g[j] = rr[j] > 0.f ? g[j] : 0.f;
    }
    float o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = k[j] * (g[j] - sg[j] - (xx[j] - mu[j]) * rs[j] * sgx[j]);
    dx4[i] = make_float4(o[0], o[1], o[2], o[3]);
  }
}

__global__ void d2f_kernel(const double* __restrict__ in, float* __restrict__ out, long n, float scale) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (float)(in[i] * (double)scale);
}

// ---------------------------------------------------------------- backward-filter of a 1x1x1 conv
// dW[k, n] += sum_m A[row(m), k] * dD[m, n]; row(m) as in x3d_pw_fwd (gather for the strided
// shortcut).  One block = a TK x TN tile of dW over a run of rows; 16 x 16 threads, each a
// (TK/16) x (TN/16) register tile fed by 128-bit shared-memory reads (k and n interleaved by 16
// so that a thread's values are contiguous); fp32 partial per block, fp64 atomics.
template <int TK, int TN>
__global__ void __launch_bounds__(256)
pw_wgrad_kernel(const float* __restrict__ A, const float* __restrict__ dD, double* __restrict__ dW, long M,
                int K, int N, int lda, int ldd, long rows_per_block, int gather, int Ho, int Wo, int Hi,
                int Wi, int stride) {
  constexpr int RK = TK / 16, RN = TN / 16, RC = 32;       // register tile, rows per chunk
  // element (r, k) of the A chunk lives at sa[r][(k % 16) * RK + k / 16]: thread ty reads RK contiguous floats
  __shared__ __align__(16) float sa[RC][TK + 4];
  __shared__ __align__(16) float sd[RC][TN + 4];
  const int k0 = blockIdx.x * TK, n0 = blockIdx.y * TN;
  const long m0 = (long)blockIdx.z * rows_per_block;
  long m1 = m0 + rows_per_block;
  if (m1 > M) m1 = M;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;  // 16 x 16
  float acc[RK][RN];
#pragma unroll
  for (int i = 0; i < RK; ++i)
#pragma unroll
    for (int j = 0; j < RN; ++j) acc[i][j] = 0.f;
  for (long mb = m0; mb < m1; mb += RC) {
    // fill: 256 threads, consecutive threads -> consecutive k (n) of one row
    for (int e = threadIdx.x; e < RC * TK; e += 256) {
      const int r = e / TK, k = e - r * TK;
      const long m = mb + r;
      float v = 0.f;
      if (m < m1 && k0 + k < K) {
        long arow = m;
        if (gather) {
          long q = m;
          const int wo = (int)(q % Wo); q /= Wo;
          const int ho = (int)(q % Ho); q /= Ho;
          arow = (q * Hi + (long)ho * stride) * Wi + (long)wo * stride;
        }
        v = __ldg(A + arow * lda + k0 + k);
      }
      sa[r][(k & 15) * RK + (k >> 4)] = v;
    }
    for (int e = threadIdx.x; e < RC * TN; e += 256) {
      const int r = e / TN, nn = e - r * TN;
      const long m = mb + r;
      sd[r][(nn & 15) * RN + (nn >> 4)] = (m < m1 && n0 + nn < N) ? __ldg(dD + m * ldd + n0 + nn) : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int r = 0; r < RC; ++r) {
      float a[RK], d[RN];
      if (RK == 4) { const float4 v = *reinterpret_cast<const float4*>(&sa[r][ty * 4]); a[0] = v.x; a[1] = v.y; a[2 % RK] = v.z; a[3 % RK] = v.w; }
      else { const float2 v = *reinterpret_cast<const float2*>(&sa[r][ty * 2]); a[0] = v.x; a[1] = v.y; }
      if (RN == 4) { const float4 v = *reinterpret_cast<const float4*>(&sd[r][tx * 4]); d[0] = v.x; d[1] = v.y; d[2 % RN] = v.z; d[3 % RN] = v.w; }
      else { const float2 v = *reinterpret_cast<const float2*>(&sd[r][tx * 2]); d[0] = v.x; d[1] = v.y; }
#pragma unroll
      for (int i = 0; i < RK; ++i)
#pragma unroll
        for (int j = 0; j < RN; ++j) acc[i][j] = fmaf(a[i], d[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < RK; ++i)
#pragma unroll
    for (int j = 0; j < RN; ++j) {
      const int k = k0 + ty + 16 * i, nn = n0 + tx + 16 * j;
      if (k < K && nn < N) atomicAdd(dW + (long)k * N + nn, (double)acc[i][j]);
    }
}

// The same backward-filter on the tensor cores: dW (TK x TN tile) = A^T (k x rows) . dD (rows x n) as
// m16n8k8 TF32 MMAs with the 3xTF32 split (hi/lo TF32 halves, lo.hi + hi.lo + hi.hi), fp32
// accumulators per block, fp64 atomics at the end as above.  8 warps tile the TK x TN block; row
// chunks of 32 are double-buffered in shared memory, the next chunk is fetched (128-bit loads) while
// the MMAs of the current one run.  Needs K, N, lda, ldd multiples of 4 (training layouts pad to 8).
// hi = x rounded to TF32 (half away from zero) with integer ops, lo = x - hi (exact) pre-biased by half a
// TF32 ulp so that the tensor core's truncation of the low 13 mantissa bits rounds it.  cvt.rna.tf32
// runs on the 16-lane conversion pipe and made the kernel conversion-bound (measured: 124 MAC/clk/SM).
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi)) + 0x1000u;
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
      "{%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

template <int TK, int TN>
__global__ void __launch_bounds__(256)
pw_wgrad_tf32x3_kernel(const float* __restrict__ A, const float* __restrict__ dD, double* __restrict__ dW, long M,
                       int K, int N, int lda, int ldd, long rows_per_block, int gather, int Ho, int Wo, int Hi,
                       int Wi, int stride) {
  constexpr int RC = 32;
  constexpr int WN = (TN == 64 && TK == 32) ? 8 : 4, WK = 8 / WN;      // warp grid over the tile
  constexpr int MF = TK / (16 * WK), NF = TN / (8 * WN);               // m16 / n8 fragments per warp
  constexpr int PA = TK + 8, PD = TN + 8;                              // pitch = 8 (mod 32): conflict-free fragments
  constexpr int VA = TK / 32, VD = TN / 32;                            // float4 per thread and chunk
  __shared__ __align__(16) float sa[2][RC][PA];
  __shared__ __align__(16) float sd[2][RC][PD];
  const int k0 = blockIdx.x * TK, n0 = blockIdx.y * TN;
  const long m0 = (long)blockIdx.z * rows_per_block;
  long m1 = m0 + rows_per_block;
  if (m1 > M) m1 = M;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int wk = (warp / WN) * MF * 16, wn = (warp % WN) * NF * 8;

  float4 ra[VA], rd[VD];
  auto fetch = [&](long mb) {
#pragma unroll
    for (int v = 0; v < VA; ++v) {
      const int e = tid + v * 256, r = e / (TK / 4), k = (e % (TK / 4)) * 4;
      const long m = mb + r;
      ra[v] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m < m1 && k0 + k < K) {
        long arow = m;
        if (gather) {
          long q = m;
          const int wo = (int)(q % Wo); q /= Wo;
          const int ho = (int)(q % Ho); q /= Ho;
          arow = (q * Hi + (long)ho * stride) * Wi + (long)wo * stride;
        }
        ra[v] = __ldg(reinterpret_cast<const float4*>(A + arow * lda + k0 + k));
      }
    }
#pragma unroll
    for (int v = 0; v < VD; ++v) {
      const int e = tid + v * 256, r = e / (TN / 4), nn = (e % (TN / 4)) * 4;
      const long m = mb + r;
      rd[v] = (m < m1 && n0 + nn < N) ? __ldg(reinterpret_cast<const float4*>(dD + m * ldd + n0 + nn))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto stage = [&](int buf) {
#pragma unroll
    for (int v = 0; v < VA; ++v) {
      const int e = tid + v * 256;
      *reinterpret_cast<float4*>(&sa[buf][e / (TK / 4)][(e % (TK / 4)) * 4]) = ra[v];
    }
#pragma unroll
    for (int v = 0; v < VD; ++v) {
      const int e = tid + v * 256;
      *reinterpret_cast<float4*>(&sd[buf][e / (TN / 4)][(e % (TN / 4)) * 4]) = rd[v];
    }
  };

  // acc: running sums (round-to-nearest fp32 adds); part: the MMA accumulators of one 32-row chunk,
  // so that the tensor core's truncating accumulation never spans more than 12 MMAs
  float acc[MF][NF][4], part[MF][NF][4];
#pragma unroll
  for (int i = 0; i < MF; ++i)
#pragma unroll
    for (int j = 0; j < NF; ++j)
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[i][j][r] = part[i][j][r] = 0.f;

  fetch(m0);
  stage(0);
  __syncthreads();
  int buf = 0;
  for (long mb = m0; mb < m1; mb += RC, buf ^= 1) {
    const bool more = mb + RC < m1;
    if (more) fetch(mb + RC);
#pragma unroll
    for (int ks = 0; ks < RC; ks += 8) {
      uint32_t ah[MF][4], al[MF][4], bh[NF][2], bl[NF][2];
#pragma unroll
      for (int i = 0; i < MF; ++i) {
        const float* ap = &sa[buf][ks + t][wk + i * 16 + g];
        split_tf32(ap[0], ah[i][0], al[i][0]);
        split_tf32(ap[8], ah[i][1], al[i][1]);
        split_tf32(ap[4 * PA], ah[i][2], al[i][2]);
        split_tf32(ap[4 * PA + 8], ah[i][3], al[i][3]);
      }
#pragma unroll
      for (int j = 0; j < NF; ++j) {
        const float* bp = &sd[buf][ks + t][wn + j * 8 + g];
        split_tf32(bp[0], bh[j][0], bl[j][0]);
        split_tf32(bp[4 * PD], bh[j][1], bl[j][1]);
      }
#pragma unroll
      for (int term = 0; term < 3; ++term)       // term-major: independent MMAs between dependent ones
#pragma unroll
        for (int i = 0; i < MF; ++i)
#pragma unroll
          for (int j = 0; j < NF; ++j) mma_tf32(part[i][j], term == 0 ? al[i] : ah[i], term == 1 ? bl[j] : bh[j]);
    }
#pragma unroll
    for (int i = 0; i < MF; ++i)
#pragma unroll
      for (int j = 0; j < NF; ++j)
#pragma unroll
        for (int r = 0; r < 4; ++r) { acc[i][j][r] += part[i][j][r]; part[i][j][r] = 0.f; }
    if (more) stage(buf ^ 1);
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < MF; ++i)
#pragma unroll
    for (int j = 0; j < NF; ++j)
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int k = k0 + wk + i * 16 + g + (r >> 1) * 8, nn = n0 + wn + j * 8 + 2 * t + (r & 1);
        if (k < K && nn < N) atomicAdd(dW + (long)k * N + nn, (double)acc[i][j][r]);
      }
}

// The backward-filter of the mixed-precision step: the structure of pw_wgrad_tf32x3_kernel (same tiles,
// warp grid, double-buffered 32-row chunks and fp32 fold per chunk, fp64 atomics), with the operands
// rounded to bf16 (RNE, cvt.rn.bf16x2) and one m16n8k16 bf16 MMA where the 3xTF32 split issues three
// per k8 step.  The MMA's reduction dim is the row: a register holds two consecutive rows.
__device__ __forceinline__ uint32_t bf16x2_rn(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
      "{%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

template <int TK, int TN>
__global__ void __launch_bounds__(256)
pw_wgrad_bf16_kernel(const float* __restrict__ A, const float* __restrict__ dD, double* __restrict__ dW, long M,
                     int K, int N, int lda, int ldd, long rows_per_block, int gather, int Ho, int Wo, int Hi,
                     int Wi, int stride) {
  constexpr int RC = 32;
  constexpr int WN = (TN == 64 && TK == 32) ? 8 : 4, WK = 8 / WN;
  constexpr int MF = TK / (16 * WK), NF = TN / (8 * WN);
  constexpr int PA = TK + 8, PD = TN + 8;
  constexpr int VA = TK / 32, VD = TN / 32;
  __shared__ __align__(16) float sa[2][RC][PA];
  __shared__ __align__(16) float sd[2][RC][PD];
  const int k0 = blockIdx.x * TK, n0 = blockIdx.y * TN;
  const long m0 = (long)blockIdx.z * rows_per_block;
  long m1 = m0 + rows_per_block;
  if (m1 > M) m1 = M;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int wk = (warp / WN) * MF * 16, wn = (warp % WN) * NF * 8;

  float4 ra[VA], rd[VD];
  auto fetch = [&](long mb) {
#pragma unroll
    for (int v = 0; v < VA; ++v) {
      const int e = tid + v * 256, r = e / (TK / 4), k = (e % (TK / 4)) * 4;
      const long m = mb + r;
      ra[v] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m < m1 && k0 + k < K) {
        long arow = m;
        if (gather) {
          long q = m;
          const int wo = (int)(q % Wo); q /= Wo;
          const int ho = (int)(q % Ho); q /= Ho;
          arow = (q * Hi + (long)ho * stride) * Wi + (long)wo * stride;
        }
        ra[v] = __ldg(reinterpret_cast<const float4*>(A + arow * lda + k0 + k));
      }
    }
#pragma unroll
    for (int v = 0; v < VD; ++v) {
      const int e = tid + v * 256, r = e / (TN / 4), nn = (e % (TN / 4)) * 4;
      const long m = mb + r;
      rd[v] = (m < m1 && n0 + nn < N) ? __ldg(reinterpret_cast<const float4*>(dD + m * ldd + n0 + nn))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto stage = [&](int buf) {
#pragma unroll
    for (int v = 0; v < VA; ++v) {
      const int e = tid + v * 256;
      *reinterpret_cast<float4*>(&sa[buf][e / (TK / 4)][(e % (TK / 4)) * 4]) = ra[v];
    }
#pragma unroll
    for (int v = 0; v < VD; ++v) {
      const int e = tid + v * 256;
      *reinterpret_cast<float4*>(&sd[buf][e / (TN / 4)][(e % (TN / 4)) * 4]) = rd[v];
    }
  };

  float acc[MF][NF][4], part[MF][NF][4];
#pragma unroll
  for (int i = 0; i < MF; ++i)
#pragma unroll
    for (int j = 0; j < NF; ++j)
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[i][j][r] = part[i][j][r] = 0.f;

  fetch(m0);
  stage(0);
  __syncthreads();
  int buf = 0;
  for (long mb = m0; mb < m1; mb += RC, buf ^= 1) {
    const bool more = mb + RC < m1;
    if (more) fetch(mb + RC);
#pragma unroll
    for (int ks = 0; ks < RC; ks += 16) {
      uint32_t a[MF][4], b[NF][2];
#pragma unroll
      for (int i = 0; i < MF; ++i) {
        const float* ap = &sa[buf][ks + 2 * t][wk + i * 16 + g];
        a[i][0] = bf16x2_rn(ap[0], ap[PA]);
        a[i][1] = bf16x2_rn(ap[8], ap[PA + 8]);
        a[i][2] = bf16x2_rn(ap[8 * PA], ap[9 * PA]);
        a[i][3] = bf16x2_rn(ap[8 * PA + 8], ap[9 * PA + 8]);
      }
#pragma unroll
      for (int j = 0; j < NF; ++j) {
        const float* bp = &sd[buf][ks + 2 * t][wn + j * 8 + g];
        b[j][0] = bf16x2_rn(bp[0], bp[PD]);
        b[j][1] = bf16x2_rn(bp[8 * PD], bp[9 * PD]);
      }
#pragma unroll
      for (int i = 0; i < MF; ++i)
#pragma unroll
        for (int j = 0; j < NF; ++j) mma_bf16(part[i][j], a[i], b[j]);
    }
#pragma unroll
    for (int i = 0; i < MF; ++i)
#pragma unroll
      for (int j = 0; j < NF; ++j)
#pragma unroll
        for (int r = 0; r < 4; ++r) { acc[i][j][r] += part[i][j][r]; part[i][j][r] = 0.f; }
    if (more) stage(buf ^ 1);
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < MF; ++i)
#pragma unroll
    for (int j = 0; j < NF; ++j)
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int k = k0 + wk + i * 16 + g + (r >> 1) * 8, nn = n0 + wn + j * 8 + 2 * t + (r & 1);
        if (k < K && nn < N) atomicAdd(dW + (long)k * N + nn, (double)acc[i][j][r]);
      }
}

// ---------------------------------------------------------------- channelwise 3x3x3 backward
// backward-data (gather form): dx[n,t,h,w,c] = sum_taps dy[n, t+1-dt, (h+ph-dh)/s, (w+pw-dw)/s, c] * w[tap,c]
__global__ void __launch_bounds__(256)
dw_dgrad_kernel(const float* __restrict__ dy, const float* __restrict__ w, float* __restrict__ dx, int T, int H,
                int W, int Ho, int Wo, int C, int stride, int ph, int pw, long total) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    long q = i / C;
    const int x = (int)(q % W); q /= W;
    const int y = (int)(q % H); q /= H;
    const int t = (int)(q % T);
    const long n = q / T;
    float acc = 0.f;
    for (int dt = 0; dt < 3; ++dt) {
      const int to = t + 1 - dt;
      if (to < 0 || to >= T) continue;
      for (int dh = 0; dh < 3; ++dh) {
        const int hy = y + ph - dh;
        if (hy < 0 || hy % stride) continue;
        const int ho = hy / stride;
        if (ho >= Ho) continue;
        for (int dw = 0; dw < 3; ++dw) {
          const int wx = x + pw - dw;
          if (wx < 0 || wx % stride) continue;
          const int wo = wx / stride;
          if (wo >= Wo) continue;
          acc = fmaf(dy[(((n * T + to) * Ho + ho) * (long)Wo + wo) * C + c], w[((dt * 3 + dh) * 3 + dw) * C + c], acc);
        }
      }
    }
    dx[i] = acc;
  }
}

// Sliding-window form of the channelwise backward-filter (kept for stride 2, where the batched kernel
// below would reload 22 values per output pixel instead of 18): the 9 x 3 input window of the current
// output pixel lives in registers and slides one output pixel per step.
__global__ void __launch_bounds__(256)
dw_wgrad_slide_kernel(const float* __restrict__ x, const float* __restrict__ dy, double* __restrict__ dwt, int T, int H,
                int W, int Ho, int Wo, int C, int stride, int ph, int pw, long orows, long rows_per_block) {
  const int lane = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  const long r0 = (long)blockIdx.y * rows_per_block;
  long r1 = r0 + rows_per_block;
  if (r1 > orows) r1 = orows;
  float acc[27];
#pragma unroll
  for (int i = 0; i < 27; ++i) acc[i] = 0.f;
  if (c < C) {
    for (long row = r0 + ry; row < r1; row += 8) {
      long q = row;
      const int ho = (int)(q % Ho); q /= Ho;
      const int t = (int)(q % T);
      const long n = q / T;
      const float* src[9];                  // input rows (dt, dh) of this output row, or null
#pragma unroll
      for (int dt = 0; dt < 3; ++dt)
#pragma unroll
        for (int dh = 0; dh < 3; ++dh) {
          const int ti = t + dt - 1, hi = ho * stride + dh - ph;
          src[dt * 3 + dh] = (ti >= 0 && ti < T && hi >= 0 && hi < H)
                                 ? x + (((n * T + ti) * H + hi) * (long)W) * C + c : nullptr;
        }
      const float* g = dy + row * (long)Wo * C + c;
      float xv[9][3];
      // columns wi = wo*stride + dw - pw; prime the window for wo = 0
#pragma unroll
      for (int k = 0; k < 9; ++k)
#pragma unroll
        for (int dw = 0; dw < 3; ++dw) {
          const int wi = dw - pw;
          xv[k][dw] = (src[k] != nullptr && wi >= 0 && wi < W) ? __ldg(src[k] + (long)wi * C) : 0.f;
        }
      for (int wo = 0; wo < Wo; ++wo) {
        const float gv = __ldg(g + (long)wo * C);
#pragma unroll
        for (int k = 0; k < 9; ++k)
#pragma unroll
          for (int dw = 0; dw < 3; ++dw) acc[k * 3 + dw] = fmaf(xv[k][dw], gv, acc[k * 3 + dw]);
        if (wo + 1 < Wo) {                   // slide to the next output pixel
          const int wn = (wo + 1) * stride - pw;          // its leftmost column
          if (stride == 1) {
            const int wi = wn + 2;
            const bool ok = wi < W;
#pragma unroll
            for (int k = 0; k < 9; ++k) {
              xv[k][0] = xv[k][1]; xv[k][1] = xv[k][2];
              xv[k][2] = (ok && src[k] != nullptr) ? __ldg(src[k] + (long)wi * C) : 0.f;
            }
          } else {
            const bool ok1 = wn + 1 < W, ok2 = wn + 2 < W;
#pragma unroll
            for (int k = 0; k < 9; ++k) {
              xv[k][0] = xv[k][2];
              xv[k][1] = (ok1 && src[k] != nullptr) ? __ldg(src[k] + (long)(wn + 1) * C) : 0.f;
              xv[k][2] = (ok2 && src[k] != nullptr) ? __ldg(src[k] + (long)(wn + 2) * C) : 0.f;
            }
          }
        }
      }
    }
  }
  __shared__ float sh[8][32];
  for (int tap = 0; tap < 27; ++tap) {
    sh[ry][lane] = acc[tap];
    __syncthreads();
    if (ry == 0 && c < C) {
      double s = 0.0;
      for (int i = 0; i < 8; ++i) s += sh[i][lane];
      atomicAdd(dwt + (long)tap * C + c, s);
    }
    __syncthreads();
  }
}

// backward-filter: dw[tap,c] += sum over output pixels x[n, t+dt-1, ho*s+dh-ph, wo*s+dw-pw, c] * dy[n,t,ho,wo,c]
// A warp (32 consecutive channels, coalesced 128-byte rows) walks whole output rows (n, t, ho) left to
// right, U output pixels per step: the 9 x ((U-1)*S+3) input values and the U dy values of a step are
// independent loads issued together (one memory round trip per step; the first version slid a 9x3
// window one pixel at a time and paid one round trip per pixel: 170 us for a 43 MB stage-5 layer),
// then 27*U FMAs.  Row validity (temporal / vertical zero padding) is resolved once per row.  The 27
// per-warp sums meet in shared memory once per block; fp64 atomics.
template <int S, int U>
__global__ void __launch_bounds__(256, 2)
dw_wgrad_kernel(const float* __restrict__ x, const float* __restrict__ dy, double* __restrict__ dwt, int T, int H,
                int W, int Ho, int Wo, int C, int ph, int pw, long orows, long rows_per_block) {
  constexpr int NC = (U - 1) * S + 3;
  const int lane = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  const long r0 = (long)blockIdx.y * rows_per_block;
  long r1 = r0 + rows_per_block;
  if (r1 > orows) r1 = orows;
  float acc[27];
#pragma unroll
  for (int i = 0; i < 27; ++i) acc[i] = 0.f;
  if (c < C) {
    for (long row = r0 + ry; row < r1; row += 8) {
      long q = row;
      const int ho = (int)(q % Ho); q /= Ho;
      const int t = (int)(q % T);
      const long n = q / T;
      const float* src[9];                  // input rows (dt, dh) of this output row, or null
#pragma unroll
      for (int dt = 0; dt < 3; ++dt)
#pragma unroll
        for (int dh = 0; dh < 3; ++dh) {
          const int ti = t + dt - 1, hi = ho * S + dh - ph;
          src[dt * 3 + dh] = (ti >= 0 && ti < T && hi >= 0 && hi < H)
                                 ? x + (((n * T + ti) * H + hi) * (long)W) * C + c : nullptr;
        }
      const float* g = dy + row * (long)Wo * C + c;
      for (int wo0 = 0; wo0 < Wo; wo0 += U) {
        const int wi0 = wo0 * S - pw;
        // column offsets (clamped into the row) and validity: warp-uniform, once per step, so that a
        // load costs one address add and one select (ncu: the first version spent 9 instructions
        // per FMA on predicated 64-bit addressing)
        int off[NC];
        bool ok[NC];
#pragma unroll
        for (int j = 0; j < NC; ++j) {
          const int wi = wi0 + j;
          ok[j] = wi >= 0 && wi < W;
          off[j] = min(max(wi, 0), W - 1) * C;
        }
        float xv[9][NC], gv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) gv[u] = (wo0 + u < Wo) ? __ldg(g + (wo0 + u) * C) : 0.f;
#pragma unroll
        for (int k = 0; k < 9; ++k) {
          if (src[k] != nullptr) {            // uniform: depends on (t, ho) only
#pragma unroll
            for (int j = 0; j < NC; ++j) {
              const float v = __ldg(src[k] + off[j]);
              xv[k][j] = ok[j] ? v : 0.f;
            }
          } else {
#pragma unroll
            for (int j = 0; j < NC; ++j) xv[k][j] = 0.f;
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
          for (int k = 0; k < 9; ++k)
#pragma unroll
            for (int dw = 0; dw < 3; ++dw) acc[k * 3 + dw] = fmaf(xv[k][u * S + dw], gv[u], acc[k * 3 + dw]);
      }
    }
  }
  __shared__ float sh[8][27][32];
#pragma unroll
  for (int tap = 0; tap < 27; ++tap) sh[ry][tap][lane] = acc[tap];
  __syncthreads();
  for (int e = threadIdx.x; e < 27 * 32; e += 256) {
    const int tap = e >> 5, l = e & 31;
    if (blockIdx.x * 32 + l >= C) continue;
    double sum = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) sum += sh[i][tap][l];
    atomicAdd(dwt + (long)tap * C + blockIdx.x * 32 + l, sum);
  }
}

// ---------------------------------------------------------------- stem pieces (training form)
// conv_s: 1x3x3, stride (1,2,2), explicit zero pad 1 on H and W, 3 -> C (model.py:161-184,203-204)
// One thread = one output pixel x 4 channels (128-bit weight loads and stores); blockIdx.x = output
// row (n*T*Ho + ho), so the only per-element division left is by the small C/4.
__global__ void __launch_bounds__(256)
stem_convs_fwd_kernel(const float* __restrict__ in, const float* __restrict__ ws, float* __restrict__ out, int H,
                      int W, int Ho, int Wo, int C) {
  const int C4 = C >> 2;
  const long row = blockIdx.x;
  const int ho = (int)(row % Ho);
  const long nt = row / Ho;
  for (int e = threadIdx.x; e < Wo * C4; e += blockDim.x) {
    const int wo = e / C4, c = (e - wo * C4) << 2;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int dh = 0; dh < 3; ++dh) {
      const int hi = 2 * ho + dh - 1;
      if (hi < 0 || hi >= H) continue;
#pragma unroll
      for (int dw = 0; dw < 3; ++dw) {
        const int wi = 2 * wo + dw - 1;
        if (wi < 0 || wi >= W) continue;
        const float* px = in + ((nt * H + hi) * (long)W + wi) * 3;
        const float* wk = ws + ((dh * 3 + dw) * 3) * C + c;
#pragma unroll
        for (int ci = 0; ci < 3; ++ci) {
          const float x = __ldg(px + ci);
          const float4 w = __ldg(reinterpret_cast<const float4*>(wk + ci * C));
          acc.x = fmaf(x, w.x, acc.x); acc.y = fmaf(x, w.y, acc.y);
          acc.z = fmaf(x, w.z, acc.z); acc.w = fmaf(x, w.w, acc.w);
        }
      }
    }
    *reinterpret_cast<float4*>(out + (row * Wo + wo) * (long)C + c) = acc;
  }
}
// backward-filter of conv_s: dws[(dh*3+dw)*3+ci, c] += sum in[...] * ds[n,t,ho,wo,c]
__global__ void __launch_bounds__(256)
stem_convs_wgrad_kernel(const float* __restrict__ in, const float* __restrict__ ds, double* __restrict__ dws, int H,
                        int W, int Ho, int Wo, int C, long opix, long pix_per_block) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ry = threadIdx.x >> 5;
  const long p0 = (long)blockIdx.y * pix_per_block;
  long p1 = p0 + pix_per_block;
  if (p1 > opix) p1 = opix;
  float acc[27];
#pragma unroll
  for (int i = 0; i < 27; ++i) acc[i] = 0.f;
  if (c < C) {
    for (long p = p0 + ry; p < p1; p += 8) {
      long q = p;
      const int wo = (int)(q % Wo); q /= Wo;
      const int ho = (int)(q % Ho);
      const long nt = q / Ho;
      const float g = ds[p * C + c];
#pragma unroll
      for (int dh = 0; dh < 3; ++dh) {
        const int hi = 2 * ho + dh - 1;
#pragma unroll
        for (int dw = 0; dw < 3; ++dw) {
          const int wi = 2 * wo + dw - 1;
          if (hi >= 0 && hi < H && wi >= 0 && wi < W) {
            const float* px = in + ((nt * H + hi) * (long)W + wi) * 3;
#pragma unroll
            for (int ci = 0; ci < 3; ++ci) acc[(dh * 3 + dw) * 3 + ci] = fmaf(px[ci], g, acc[(dh * 3 + dw) * 3 + ci]);
          }
        }
      }
    }
  }
  __shared__ float sh[8][32];
  for (int k = 0; k < 27; ++k) {
    sh[ry][threadIdx.x & 31] = acc[k];
    __syncthreads();
    if (ry == 0 && c < C) {
      double s = 0.0;
      for (int i = 0; i < 8; ++i) s += sh[i][threadIdx.x];
      atomicAdd(dws + (long)k * C + c, s);
    }
    __syncthreads();
  }
}
// conv_t: kt x1x1 channelwise over T with zero pad kt/2 (model.py:170-175,187-194,205-206).
// out[n,t,p,c] = sum_d in[n, t+d-kt/2, p, c] * wt[d',c],  d' = flip ? kt-1-d : d  (flip = backward-data)
// One thread = 4 channels of one pixel; a block works inside one frame (n*T + t): 128-bit loads, one
// small modulo per element instead of three 64-bit divisions.
__global__ void __launch_bounds__(256)
tconv_fwd_kernel(const float* __restrict__ in, const float* __restrict__ wt, float* __restrict__ out, int T,
                 long P, int C, int kt, int flip, int blocks_per_frame) {
  const int C4 = C >> 2;
  const long frame4 = P * C4;                       // float4 elements per frame
  const long nt = blockIdx.x / blocks_per_frame;
  const int bx = blockIdx.x - (int)(nt * blocks_per_frame);
  const int t = (int)(nt % T);
  const float4* in4 = reinterpret_cast<const float4*>(in);
  float4* out4 = reinterpret_cast<float4*>(out);
  for (long e = (long)bx * blockDim.x + threadIdx.x; e < frame4; e += (long)blocks_per_frame * blockDim.x) {
    const int c = (int)(e % C4) << 2;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int d = 0; d < kt; ++d) {
      const int ti = t + d - kt / 2;
      if (ti < 0 || ti >= T) continue;
      const float4 x = __ldg(in4 + (nt + d - kt / 2) * frame4 + e);
      const float4 w = __ldg(reinterpret_cast<const float4*>(wt + (flip ? kt - 1 - d : d) * C + c));
      acc.x = fmaf(x.x, w.x, acc.x); acc.y = fmaf(x.y, w.y, acc.y);
      acc.z = fmaf(x.z, w.z, acc.z); acc.w = fmaf(x.w, w.w, acc.w);
    }
    out4[nt * frame4 + e] = acc;
  }
}
// dwt[d,c] += sum s[n, t+d-kt/2, p, c] * dy[n,t,p,c]
__global__ void __launch_bounds__(256)
tconv_wgrad_kernel(const float* __restrict__ s, const float* __restrict__ dy, double* __restrict__ dwt, int T,
                   long P, int C, int kt, long rows, long rows_per_block) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ry = threadIdx.x >> 5;
  const long r0 = (long)blockIdx.y * rows_per_block;
  long r1 = r0 + rows_per_block;
  if (r1 > rows) r1 = rows;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  if (c < C) {
    for (long r = r0 + ry; r < r1; r += 8) {      // r = (n*T + t)*P + p
      const long nt = r / P, pp = r % P;
      const int t = (int)(nt % T);
      const float g = dy[r * C + c];
      for (int d = 0; d < kt; ++d) {
        const int ti = t + d - kt / 2;
        if (ti >= 0 && ti < T) acc[d] = fmaf(s[((nt - t + ti) * P + pp) * C + c], g, acc[d]);
      }
    }
  }
  __shared__ float sh[8][32];
  for (int d = 0; d < kt; ++d) {
    sh[ry][threadIdx.x & 31] = acc[d];
    __syncthreads();
    if (ry == 0 && c < C) {
      double sum = 0.0;
      for (int i = 0; i < 8; ++i) sum += sh[i][threadIdx.x];
      atomicAdd(dwt + (long)d * C + c, sum);
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------- elementwise pieces
__device__ __forceinline__ float sigm(float x) { return 1.f / (1.f + expf(-x)); }

// out = swish(y * s[n, c])   (s == nullptr: factor 1)      model.py:311-316
__global__ void __launch_bounds__(256)
scale_swish_fwd_kernel(const float* __restrict__ y, const float* __restrict__ s, float* __restrict__ out,
                       long clip4, int C4, long stride4) {
  // blockIdx.y = clip; 128-bit accesses; the thread stride is a multiple of C/4, so a thread keeps its
  // 4 channels (and their SE factors) for the whole clip
  const long i0 = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i0 >= clip4 || i0 >= stride4) return;
  const long n = blockIdx.y;
  const int c = (int)(i0 % C4) << 2;
  float sc[4] = {1.f, 1.f, 1.f, 1.f};
  if (s) {
#pragma unroll
    for (int j = 0; j < 4; ++j) sc[j] = s[n * (C4 << 2) + c + j];
  }
  const float4* y4 = reinterpret_cast<const float4*>(y) + n * clip4;
  float4* o4 = reinterpret_cast<float4*>(out) + n * clip4;
  for (long i = i0; i < clip4; i += stride4) {
    const float4 v = __ldg(y4 + i);
    const float a[4] = {v.x * sc[0], v.y * sc[1], v.z * sc[2], v.w * sc[3]};
    o4[i] = make_float4(a[0] * sigm(a[0]), a[1] * sigm(a[1]), a[2] * sigm(a[2]), a[3] * sigm(a[3]));
  }
}
// dv = dout * (sig(v) * (1 + v * (1 - sig(v))));  dy = dv * s;  ds[n,c] += sum_p dv * y
__global__ void __launch_bounds__(256)
scale_swish_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ y, const float* __restrict__ s,
                       float* __restrict__ dy, double* __restrict__ ds, int C, long rows_per_clip) {
  // grid: (ceil(C/32), row blocks of the clip, clips)
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ry = threadIdx.x >> 5;
  const long n = blockIdx.z;
  const long r0 = n * rows_per_clip + (long)blockIdx.y * kRowsPerBlock;
  long r1 = r0 + kRowsPerBlock;
  if (r1 > (n + 1) * rows_per_clip) r1 = (n + 1) * rows_per_clip;
  float acc = 0.f;
  if (c < C) {
    const float sc = s ? s[n * C + c] : 1.f;
    for (long r = r0 + ry; r < r1; r += 8) {
      const float yv = y[r * C + c], v = yv * sc, sg = sigm(v);
      const float dv = dout[r * C + c] * (sg * (1.f + v * (1.f - sg)));
      dy[r * C + c] = dv * sc;
      acc = fmaf(dv, yv, acc);
    }
  }
  if (ds == nullptr) return;
  __shared__ float sh[8][32];
  sh[ry][threadIdx.x & 31] = acc;
  __syncthreads();
  if (ry == 0 && c < C) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += sh[i][threadIdx.x];
    atomicAdd(ds + n * C + c, t);
  }
}
// generic elementwise ops on flat arrays
//  0: out = relu(a + b)                 (ResBlock add + ReLU, model.py:389-392)
//  1: out = a * (b > 0)                 (ReLU backward, b = forward output)
//  2: out = sigmoid(a)                  3: out = a * b * (1 - b)   (sigmoid backward, b = forward output)
//  4: out = a + b                       5: out = a * b             (dropout with a precomputed mask)
__global__ void __launch_bounds__(256)
ew_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, long n, int op) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float x = a[i], y = b ? b[i] : 0.f;
    float r;
    switch (op) {
      case 0: r = fmaxf(x + y, 0.f); break;
      case 1: r = y > 0.f ? x : 0.f; break;
      case 2: r = sigm(x); break;
      case 3: r = x * y * (1.f - y); break;
      case 4: r = x + y; break;
      default: r = x * y; break;
    }
    out[i] = r;
  }
}
// dy[n, p, c] (+)= dm[n, c] * scale     (backward of the global average pool, scale = 1/P)
__global__ void __launch_bounds__(256)
pool_bwd_kernel(const float* __restrict__ dm, float* __restrict__ dy, long total, int C, long rows_per_clip,
                float scale, int accumulate) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const float v = dm[(i / C / rows_per_clip) * C + (i % C)] * scale;
    dy[i] = accumulate ? dy[i] + v : v;
  }
}
// dst[n,t,ho*s,wo*s,c] += src[n,t,ho,wo,c]   (backward-data of the strided 'valid' shortcut conv)
__global__ void __launch_bounds__(256)
strided_add_kernel(const float* __restrict__ src, float* __restrict__ dst, int Ho, int Wo, int Hi, int Wi,
                   int stride, int C, long total) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    long q = i / C;
    const int wo = (int)(q % Wo); q /= Wo;
    const int ho = (int)(q % Ho);
    const long nt = q / Ho;
    dst[((nt * Hi + (long)ho * stride) * Wi + (long)wo * stride) * C + c] += src[i];
  }
}
// dropout mask (keep with probability 1-rate, scaled by 1/(1-rate)); counter-based hash RNG
__global__ void dropout_mask_kernel(float* __restrict__ mask, long n, float rate, unsigned long long seed) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(i + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  const float u = (float)(z >> 40) * (1.f / 16777216.f);
  mask[i] = u >= rate ? 1.f / (1.f - rate) : 0.f;
}
// softmax + sparse categorical cross-entropy on the probabilities (train.py:104; Keras clips p to
// [1e-7, 1-1e-7]) and its gradient w.r.t. the logits, scaled by `gscale` (1 / global batch).
__global__ void __launch_bounds__(256)
softmax_xent_kernel(const float* __restrict__ logits, const int* __restrict__ labels, float* __restrict__ loss,
                    float* __restrict__ dlogits, int ncls, float gscale) {
  __shared__ float sh[8];
  const int n = blockIdx.x;
  const float* row = logits + (long)n * ncls;
  float m = -INFINITY;
  for (int c = threadIdx.x; c < ncls; c += blockDim.x) m = fmaxf(m, row[c]);
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
  __syncthreads();
  m = sh[0];
  for (int i = 1; i < (int)(blockDim.x >> 5); ++i) m = fmaxf(m, sh[i]);
  __syncthreads();
  float s = 0.f;
  for (int c = threadIdx.x; c < ncls; c += blockDim.x) s += expf(row[c] - m);
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  s = 0.f;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += sh[i];
  const int y = labels[n];
  const float py = expf(row[y] - m) / s;
  // d(-log(clip(p_y)))/dlogit_c = (p_c - [c==y]) when p_y is inside the clip range, else 0
  const bool inside = py > 1e-7f && py < 1.f - 1e-7f;
  for (int c = threadIdx.x; c < ncls; c += blockDim.x) {
    const float pc = expf(row[c] - m) / s;
    dlogits[(long)n * ncls + c] = inside ? (pc - (c == y ? 1.f : 0.f)) * gscale : 0.f;
  }
  if (threadIdx.x == 0) loss[n] = -logf(fminf(fmaxf(py, 1e-7f), 1.f - 1e-7f));
}
// SGD with Nesterov momentum and L2 (train.py:88-92; Keras: v = mu*v - lr*g; w += mu*v - lr*g),
// g = grad + wd[i] * w  (wd = 2 * WEIGHT_DECAY on regularised kernels, 0 elsewhere; model.py:47)
__global__ void __launch_bounds__(256)
sgd_nesterov_kernel(float* __restrict__ w, const float* __restrict__ grad, float* __restrict__ v,
                    const float* __restrict__ wd, long n, float lr, float mu) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float g = grad[i] + wd[i] * w[i];
    const float vn = mu * v[i] - lr * g;
    v[i] = vn;
    w[i] = w[i] + mu * vn - lr * g;
  }
}

// Adam as Keras applies it (train.py:93-95; tf.optimizers.Adam defaults beta_1 0.9, beta_2 0.999,
// epsilon 1e-7):  m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;  w -= lr_t m / (sqrt(v) + eps),
// lr_t = lr sqrt(1 - b2^t) / (1 - b1^t) computed by the caller;  g = grad + wd[i] w as for SGD.
__global__ void __launch_bounds__(256)
adam_kernel(float* __restrict__ w, const float* __restrict__ grad, float* __restrict__ m, float* __restrict__ v,
            const float* __restrict__ wd, long n, float lr_t, float b1, float b2, float eps) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float g = grad[i] + wd[i] * w[i];
    const float mn = b1 * m[i] + (1.f - b1) * g;
    const float vn = b2 * v[i] + (1.f - b2) * g * g;
    m[i] = mn;
    v[i] = vn;
    w[i] = w[i] - lr_t * mn / (sqrtf(vn) + eps);
  }
}

static inline unsigned ew_blocks(long n) {
  long b = (n + 255) / 256;
  if (b > 148L * 32) b = 148L * 32;
  if (b < 1) b = 1;
  return (unsigned)b;
}

}  // namespace train
}  // namespace x3d

using namespace x3d;
namespace x3d {
namespace train {
// Backward-filter of the stem's temporal conv as a stream over (pixel, channel quad) columns: a thread
// walks the T frames of its column with the KT s-values of the window in registers, so s and dy are
// each read once with 128-bit loads (the kernel above re-reads s KT times with 4-byte loads and 24 of
// 32 lanes busy at C = 24).  The block size is a multiple of C/4, a thread keeps its channel quad;
// per-thread fp32 sums are combined in fixed order in shared memory, fp64 atomics per block.
template <int KT>
__global__ void __launch_bounds__(256)
tconv_wgrad_vec_kernel(const float4* __restrict__ s, const float4* __restrict__ dy, double* __restrict__ dwt, int T,
                       long PC4, int C4, long ncols) {
  __shared__ float4 sh[KT][256];
  const int tid = threadIdx.x, bs = blockDim.x;
  float4 acc[KT];
#pragma unroll
  for (int d = 0; d < KT; ++d) acc[d] = make_float4(0.f, 0.f, 0.f, 0.f);
  const long stride = (long)gridDim.x * bs;
  for (long col = (long)blockIdx.x * bs + tid; col < ncols; col += stride) {
    const long n = col / PC4, rem = col - n * PC4;
    const float4* sp = s + n * T * PC4 + rem;
    const float4* gp = dy + n * T * PC4 + rem;
    float4 w[KT];                                         // w[d] = s[t + d - KT/2], zero outside the clip
#pragma unroll
    for (int d = 0; d < KT; ++d) {
      const int ti = d - KT / 2;
      w[d] = (ti >= 0 && ti < T) ? __ldg(sp + ti * PC4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (int t = 0; t < T; ++t) {
      const float4 g = __ldg(gp + t * PC4);
      const int tn = t + 1 + KT / 2;
      const float4 nx = tn < T ? __ldg(sp + tn * PC4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int d = 0; d < KT; ++d) {
        acc[d].x = fmaf(w[d].x, g.x, acc[d].x); acc[d].y = fmaf(w[d].y, g.y, acc[d].y);
        acc[d].z = fmaf(w[d].z, g.z, acc[d].z); acc[d].w = fmaf(w[d].w, g.w, acc[d].w);
      }
#pragma unroll
      for (int d = 0; d + 1 < KT; ++d) w[d] = w[d + 1];
      w[KT - 1] = nx;
    }
  }
#pragma unroll
  for (int d = 0; d < KT; ++d) sh[d][tid] = acc[d];
  __syncthreads();
  const int C = C4 * 4;
  for (int e = tid; e < KT * C4; e += bs) {
    const int d = e / C4, c4 = e - d * C4;
    double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0;
    for (int g = c4; g < bs; g += C4) {
      const float4 v = sh[d][g];
      t0 += v.x; t1 += v.y; t2 += v.z; t3 += v.w;
    }
    double* o = dwt + (long)d * C + c4 * 4;
    atomicAdd(o, t0); atomicAdd(o + 1, t1); atomicAdd(o + 2, t2); atomicAdd(o + 3, t3);
  }
}
}  // namespace train
}  // namespace x3d

namespace x3d {
namespace train {
// Backward-filter of the stem's spatial conv, one thread per (output pixel, channel quad): the 27 input
// values of the pixel's window meet a 128-bit load of ds, 108 FMAs per 28 loads, all lanes busy for any
// C % 4 == 0 (the kernel above keeps a warp on 32 channels of one pixel: 24 of 32 lanes at C = 24 and
// one FMA per load).  Block size a multiple of C/4; the 27 x 4 per-thread sums are combined through
// shared memory in three passes of 9 taps, fixed order, fp64 atomics per block.
__global__ void __launch_bounds__(256)
stem_convs_wgrad_vec_kernel(const float* __restrict__ in, const float4* __restrict__ ds, double* __restrict__ dws,
                            int H, int W, int Ho, int Wo, int C4, int opix) {
  __shared__ float4 sh[9][256];
  const int tid = threadIdx.x, bs = blockDim.x, ppb = bs / C4;
  const int c4 = tid % C4, pl = tid / C4;
  float4 acc[27];
#pragma unroll
  for (int k = 0; k < 27; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int p = blockIdx.x * ppb + pl; p < opix; p += gridDim.x * ppb) {
    const int wo = p % Wo, q = p / Wo;
    const int ho = q % Ho, nt = q / Ho;
    const float4 g = __ldg(ds + (long)p * C4 + c4);
    const int hi0 = 2 * ho - 1, wi0 = 2 * wo - 1;
    const float* base = in + ((long)nt * H * W) * 3;
#pragma unroll
    for (int dh = 0; dh < 3; ++dh) {
      const int hi = hi0 + dh;
      const bool rok = hi >= 0 && hi < H;
      const float* row = base + ((long)(rok ? hi : 0) * W) * 3;
#pragma unroll
      for (int dw = 0; dw < 3; ++dw) {
        const int wi = wi0 + dw;
        const bool ok = rok && wi >= 0 && wi < W;
        const float* px = row + (ok ? wi : 0) * 3;
#pragma unroll
        for (int ci = 0; ci < 3; ++ci) {
          const float v = ok ? __ldg(px + ci) : 0.f;
          float4& a = acc[(dh * 3 + dw) * 3 + ci];
          a.x = fmaf(v, g.x, a.x); a.y = fmaf(v, g.y, a.y); a.z = fmaf(v, g.z, a.z); a.w = fmaf(v, g.w, a.w);
        }
      }
    }
  }
  const int C = C4 * 4;
#pragma unroll
  for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
    for (int k = 0; k < 9; ++k) sh[k][tid] = acc[pass * 9 + k];
    __syncthreads();
    for (int e = tid; e < 9 * C4; e += bs) {
      const int k = e / C4, cc = e - k * C4;
      double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0;
      for (int gidx = cc; gidx < ppb * C4; gidx += C4) {
        const float4 v = sh[k][gidx];
        t0 += v.x; t1 += v.y; t2 += v.z; t3 += v.w;
      }
      double* o = dws + (long)(pass * 9 + k) * C + cc * 4;
      atomicAdd(o, t0); atomicAdd(o + 1, t1); atomicAdd(o + 2, t2); atomicAdd(o + 3, t3);
    }
    __syncthreads();
  }
}
}  // namespace train
}  // namespace x3d

namespace x3d {
namespace train {
// Backward of swish(y * s) as a 128-bit stream per clip: block size a multiple of C/4, a thread keeps
// its channel quad while it strides through the clip's [rows, C/4] float4 matrix; the per-clip sums
// for the SE scale's gradient are combined in shared memory in fixed order, fp64 atomics per block.
__global__ void __launch_bounds__(256)
scale_swish_bwd_vec_kernel(const float4* __restrict__ dout, const float4* __restrict__ y, const float* __restrict__ s,
                           float4* __restrict__ dy, double* __restrict__ ds, int C4, long clip4) {
  __shared__ float4 sh[256];
  const int tid = threadIdx.x, bs = blockDim.x, c4 = tid % C4;
  const long n = blockIdx.y, base = n * clip4;
  float4 sc = make_float4(1.f, 1.f, 1.f, 1.f);
  if (s) sc = __ldg(reinterpret_cast<const float4*>(s + n * C4 * 4) + c4);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  const long stride = (long)gridDim.x * bs;
#pragma unroll 2
  for (long i = (long)blockIdx.x * bs + tid; i < clip4; i += stride) {
    const float4 yv = __ldg(y + base + i), g = __ldg(dout + base + i);
    float4 o;
#define X3D_SSB(f)                                                     \
    {                                                                  \
      const float v = yv.f * sc.f, sg = sigm(v);                       \
      const float dv = g.f * (sg * (1.f + v * (1.f - sg)));            \
      o.f = dv * sc.f;                                                 \
      acc.f = fmaf(dv, yv.f, acc.f);                                   \
    }
    X3D_SSB(x) X3D_SSB(y) X3D_SSB(z) X3D_SSB(w)
#undef X3D_SSB
    dy[base + i] = o;
  }
  if (ds == nullptr) return;
  sh[tid] = acc;
  __syncthreads();
  if (tid < C4) {
    double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0;
    for (int gi = tid; gi < bs; gi += C4) {
      const float4 v = sh[gi];
      t0 += v.x; t1 += v.y; t2 += v.z; t3 += v.w;
    }
    double* o = ds + n * C4 * 4 + tid * 4;
    atomicAdd(o, t0); atomicAdd(o + 1, t1); atomicAdd(o + 2, t2); atomicAdd(o + 3, t3);
  }
}
}  // namespace train
}  // namespace x3d

namespace x3d {
namespace train {
// Channelwise backward-filter, stride 1, two channels per thread: block size a multiple of C/2, thread
// t owns channel pair t % (C/2) and row lane t / (C/2).  Per step of U = 4 output pixels the nine
// (dt, dh) input rows are visited one after the other: six 64-bit loads (clamped offsets, zero select)
// and 24 FMA pairs each, i.e. 3.7 FMAs per load against 1.9 in the one-channel kernel, with all lanes
// busy for any even C.  The 27 x 2 sums per thread are combined through shared memory in three
// passes of nine taps, fixed order; fp64 atomics per block.
__global__ void __launch_bounds__(256, 2)
dw_wgrad_pair_kernel(const float2* __restrict__ x, const float2* __restrict__ dy, double* __restrict__ dwt, int T,
                     int H, int W, int C2, int ph, int pw, int orows, int rows_per_block) {
  constexpr int U = 4, NC = U + 2;
  __shared__ float2 sh[9][256];
  const int tid = threadIdx.x, bs = blockDim.x;
  const int c2 = tid % C2, rl = tid / C2, RL = bs / C2;
  const int r0 = blockIdx.x * rows_per_block;
  const int r1 = min(r0 + rows_per_block, orows);
  float2 acc[27];
#pragma unroll
  for (int i = 0; i < 27; ++i) acc[i] = make_float2(0.f, 0.f);
  for (int row = r0 + rl; row < r1; row += RL) {
    const int ho = row % H, q = row / H;
    const int t = q % T, n = q / T;
    int src[9];                                           // float2 index of (row, column 0, c2); -1 = padding
#pragma unroll
    for (int dt = 0; dt < 3; ++dt)
#pragma unroll
      for (int dh = 0; dh < 3; ++dh) {
        const int ti = t + dt - 1, hi = ho + dh - ph;
        src[dt * 3 + dh] = (ti >= 0 && ti < T && hi >= 0 && hi < H) ? (((n * T + ti) * H + hi) * W) * C2 + c2 : -1;
      }
    const float2* g = dy + (long)row * W * C2 + c2;
    for (int wo0 = 0; wo0 < W; wo0 += U) {
      int off[NC];
      bool ok[NC];
#pragma unroll
      for (int j = 0; j < NC; ++j) {
        const int wi = wo0 - pw + j;
        ok[j] = wi >= 0 && wi < W;
        off[j] = min(max(wi, 0), W - 1) * C2;
      }
      float2 gv[U];
#pragma unroll
      for (int u = 0; u < U; ++u) gv[u] = (wo0 + u < W) ? __ldg(g + (wo0 + u) * C2) : make_float2(0.f, 0.f);
#pragma unroll
      for (int k = 0; k < 9; ++k) {
        if (src[k] < 0) continue;                         // whole input row is padding
        float2 xv[NC];
#pragma unroll
        for (int j = 0; j < NC; ++j) {
          const float2 v = __ldg(x + src[k] + off[j]);
          xv[j] = ok[j] ? v : make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
          for (int dw = 0; dw < 3; ++dw) {
            acc[k * 3 + dw].x = fmaf(xv[u + dw].x, gv[u].x, acc[k * 3 + dw].x);
            acc[k * 3 + dw].y = fmaf(xv[u + dw].y, gv[u].y, acc[k * 3 + dw].y);
          }
      }
    }
  }
  const int C = C2 * 2;
#pragma unroll
  for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
    for (int k = 0; k < 9; ++k) sh[k][tid] = acc[pass * 9 + k];
    __syncthreads();
    for (int e = tid; e < 9 * C2; e += bs) {
      const int k = e / C2, cc = e - k * C2;
      double t0 = 0.0, t1 = 0.0;
      for (int gi = cc; gi < RL * C2; gi += C2) {
        const float2 v = sh[k][gi];
        t0 += v.x; t1 += v.y;
      }
      double* o = dwt + (long)(pass * 9 + k) * C + cc * 2;
      atomicAdd(o, t0); atomicAdd(o + 1, t1);
    }
    __syncthreads();
  }
}
}  // namespace train
}  // namespace x3d

using namespace x3d::train;

extern "C" {

// Grid whose total thread count is a multiple of C/4, so that thread i always sees channel group
// i mod (C/4) when it strides through the [M, C/4] float4 matrix.
struct BnGrid { unsigned blocks; long total4, stride4; };
static BnGrid bn_grid(long M, int C, int ctas_per_sm = 8) {
  const long C4 = C / 4, total4 = M * C4;
  long threads = 148L * ctas_per_sm * 256;
  if (threads > total4) threads = total4;
  threads = (threads + C4 - 1) / C4 * C4;              // multiple of C4 ...
  long blocks = (threads + 255) / 256;
  // ... and of 256 where possible: stride = the multiple of C4 actually covered by `blocks` blocks
  const long stride4 = blocks * 256 / C4 * C4;         // threads >= stride4 never start (i0 check below)
  return BnGrid{(unsigned)blocks, total4, stride4 > 0 ? stride4 : C4};
}

int x3d_colreduce(const float* a, const float* x, const float* mean, const float* rstd, const float* relu_out,
                  int64_t M, int C, int64_t seg_rows, double* out, int mode, void* stream) {
  X3D_REQUIRE(a && out && M > 0 && C > 0 && seg_rows > 0 && mode >= 0 && mode <= 2, X3D_ERR_INVALID_ARG, "x3d_colreduce: bad argument");
  X3D_REQUIRE(mode != 1 || (x && mean && rstd), X3D_ERR_INVALID_ARG, "x3d_colreduce: mode 1 needs x, mean, rstd");
  const long segs = (M + seg_rows - 1) / seg_rows;
  if (segs == 1 && C % 4 == 0 && M * (long)(C / 4) >= 4096 &&
      ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(relu_out)) & 15) == 0) {
    const BnGrid g = bn_grid(M, C, 4);
    colreduce_vec_kernel<<<g.blocks, 256, 0, S(stream)>>>(a, x, mean, rstd, relu_out, g.total4, C / 4,
                                                                               g.stride4, out, mode);
    return check_launch("x3d_colreduce");
  }
  const long rb = (seg_rows + kRowsPerBlock - 1) / kRowsPerBlock;
  X3D_REQUIRE(segs <= 65535 && rb <= 65535, X3D_ERR_UNSUPPORTED, "x3d_colreduce: too many segments / row blocks");
  dim3 grid((C + 31) / 32, (unsigned)rb, (unsigned)segs);
  colreduce_kernel<<<grid, 256, 0, S(stream)>>>(a, x, mean, rstd, relu_out, M, C, seg_rows, out, mode);
  return check_launch("x3d_colreduce");
}

int x3d_bn_finalize(const double* sums, int64_t M, int C, float eps, float momentum, float* mean, float* var,
                    float* rstd, float* mov_mean, float* mov_var, void* stream) {
  X3D_REQUIRE(sums && mean && var && rstd && M > 0 && C > 0, X3D_ERR_INVALID_ARG, "x3d_bn_finalize: bad argument");
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, S(stream)>>>(sums, M, C, eps, momentum, mean, var, rstd, mov_mean, mov_var);
  return check_launch("x3d_bn_finalize");
}

int x3d_bn_apply_fwd(const float* x, const float* mean, const float* rstd, const float* gamma, const float* beta,
                     float* y, int64_t M, int C, int relu, void* stream) {
  X3D_REQUIRE(x && mean && rstd && gamma && beta && y && M > 0 && C > 0, X3D_ERR_INVALID_ARG, "x3d_bn_apply_fwd: bad argument");
  X3D_REQUIRE(C % 4 == 0, X3D_ERR_UNSUPPORTED, "x3d_bn_apply_fwd: C=%d must be a multiple of 4", C);
  const BnGrid g = bn_grid(M, C);
  bn_apply_kernel<<<g.blocks, 256, 0, S(stream)>>>(x, mean, rstd, gamma, beta, y, g.total4, C / 4, g.stride4, relu);
  return check_launch("x3d_bn_apply_fwd");
}

int x3d_bn_bwd_apply(const float* dy, const float* x, const float* relu_out, const float* mean, const float* rstd,
                     const float* gamma, const double* sums, float* dx, int64_t M, int C, void* stream) {
  X3D_REQUIRE(dy && x && mean && rstd && gamma && sums && dx && M > 0 && C > 0, X3D_ERR_INVALID_ARG, "x3d_bn_bwd_apply: bad argument");
  X3D_REQUIRE(C % 4 == 0, X3D_ERR_UNSUPPORTED, "x3d_bn_bwd_apply: C=%d must be a multiple of 4", C);
  const BnGrid g = bn_grid(M, C);
  bn_bwd_apply_kernel<<<g.blocks, 256, 0, S(stream)>>>(dy, x, relu_out, mean, rstd, gamma, sums, dx, g.total4, C / 4, g.stride4, M);
  return check_launch("x3d_bn_bwd_apply");
}

int x3d_d2f(const double* in, float* out, int64_t n, float scale, void* stream) {
  X3D_REQUIRE(in && out && n > 0, X3D_ERR_INVALID_ARG, "x3d_d2f: bad argument");
  d2f_kernel<<<(unsigned)((n + 255) / 256), 256, 0, S(stream)>>>(in, out, n, scale);
  return check_launch("x3d_d2f");
}

// Grid of the backward-filter kernels: TK x TN tiles of dW times row blocks of a multiple of 32 rows.
static dim3 pw_wgrad_grid(int64_t M, int K, int N, bool k64, bool n64, long& rpb) {
  const int TK = k64 ? 64 : 32, TN = n64 ? 64 : 32;
  const long tiles = (long)((K + TK - 1) / TK) * ((N + TN - 1) / TN);
  // enough row blocks for ~8 blocks per SM in total, at least 256 rows each
  long zb = (148L * 8 + tiles - 1) / tiles;
  rpb = (M + zb - 1) / zb;
  if (rpb < 256) rpb = 256;
  rpb = (rpb + 31) / 32 * 32;
  zb = (M + rpb - 1) / rpb;
  if (zb > 65535) { rpb = ((M + 65534) / 65535 + 31) / 32 * 32; zb = (M + rpb - 1) / rpb; }
  return dim3((K + TK - 1) / TK, (N + TN - 1) / TN, (unsigned)zb);
}

int x3d_pw_wgrad(const float* A, const float* dD, double* dW, int64_t M, int K, int N, int lda, int ldd, int gather,
                 int Ho, int Wo, int Hi, int Wi, int stride, void* stream) {
  X3D_REQUIRE(A && dD && dW && M > 0 && K > 0 && N > 0, X3D_ERR_INVALID_ARG, "x3d_pw_wgrad: bad argument");
  const bool k64 = K > 32, n64 = N > 32;
  long rpb;
  const dim3 grid = pw_wgrad_grid(M, K, N, k64, n64, rpb);
#define X3D_WG(TKK, TNN) train::pw_wgrad_kernel<TKK, TNN><<<grid, 256, 0, S(stream)>>>(A, dD, dW, M, K, N, lda, ldd, rpb, gather, Ho, Wo, Hi, Wi, stride)
#define X3D_WGT(TKK, TNN) train::pw_wgrad_tf32x3_kernel<TKK, TNN><<<grid, 256, 0, S(stream)>>>(A, dD, dW, M, K, N, lda, ldd, rpb, gather, Ho, Wo, Hi, Wi, stride)
  const bool vec = K % 4 == 0 && N % 4 == 0 && lda % 4 == 0 && ldd % 4 == 0 &&
                   reinterpret_cast<uintptr_t>(A) % 16 == 0 && reinterpret_cast<uintptr_t>(dD) % 16 == 0;
  if (vec) {
    if (k64 && n64) X3D_WGT(64, 64);
    else if (k64) X3D_WGT(64, 32);
    else if (n64) X3D_WGT(32, 64);
    else X3D_WGT(32, 32);
  } else {
    if (k64 && n64) X3D_WG(64, 64);
    else if (k64) X3D_WG(64, 32);
    else if (n64) X3D_WG(32, 64);
    else X3D_WG(32, 32);
  }
#undef X3D_WGT
#undef X3D_WG
  return check_launch("x3d_pw_wgrad");
}

int x3d_pw_wgrad_bf16(const float* A, const float* dD, double* dW, int64_t M, int K, int N, int lda, int ldd,
                      int gather, int Ho, int Wo, int Hi, int Wi, int stride, void* stream) {
  X3D_REQUIRE(A && dD && dW && M > 0 && K > 0 && N > 0, X3D_ERR_INVALID_ARG, "x3d_pw_wgrad_bf16: bad argument");
  X3D_REQUIRE(K % 4 == 0 && N % 4 == 0 && lda % 4 == 0 && ldd % 4 == 0 && lda >= K && ldd >= N,
              X3D_ERR_INVALID_ARG, "x3d_pw_wgrad_bf16: K=%d N=%d lda=%d ldd=%d must be multiples of 4", K, N, lda, ldd);
  X3D_REQUIRE(reinterpret_cast<uintptr_t>(A) % 16 == 0 && reinterpret_cast<uintptr_t>(dD) % 16 == 0,
              X3D_ERR_INVALID_ARG, "x3d_pw_wgrad_bf16: A and dD must be 16-byte aligned");
  X3D_REQUIRE(!gather || (Ho > 0 && Wo > 0 && Hi > 0 && Wi > 0 && stride > 0), X3D_ERR_INVALID_ARG,
              "x3d_pw_wgrad_bf16: bad gather geometry");
  const bool k64 = K > 32, n64 = N > 32;
  long rpb;
  const dim3 grid = pw_wgrad_grid(M, K, N, k64, n64, rpb);
#define X3D_WGB(TKK, TNN) train::pw_wgrad_bf16_kernel<TKK, TNN><<<grid, 256, 0, S(stream)>>>(A, dD, dW, M, K, N, lda, ldd, rpb, gather, Ho, Wo, Hi, Wi, stride)
  if (k64 && n64) X3D_WGB(64, 64);
  else if (k64) X3D_WGB(64, 32);
  else if (n64) X3D_WGB(32, 64);
  else X3D_WGB(32, 32);
#undef X3D_WGB
  return check_launch("x3d_pw_wgrad_bf16");
}

int x3d_dw_dgrad(const float* dy, const float* w, float* dx, int N, int T, int H, int W, int C, int stride, int pad_h,
                 int pad_w, void* stream) {
  X3D_REQUIRE(dy && w && dx && N > 0 && T > 0 && H > 0 && W > 0 && C > 0 && (stride == 1 || stride == 2), X3D_ERR_INVALID_ARG, "x3d_dw_dgrad: bad argument");
  const int Ho = (H + stride - 1) / stride, Wo = (W + stride - 1) / stride;
  const long total = (long)N * T * H * W * C;
  dw_dgrad_kernel<<<ew_blocks(total), 256, 0, S(stream)>>>(dy, w, dx, T, H, W, Ho, Wo, C, stride, pad_h, pad_w, total);
  return check_launch("x3d_dw_dgrad");
}

int x3d_dw_wgrad(const float* x, const float* dy, double* dwt, int N, int T, int H, int W, int C, int stride, int pad_h,
                 int pad_w, void* stream) {
  X3D_REQUIRE(x && dy && dwt && N > 0 && T > 0 && H > 0 && W > 0 && C > 0 && (stride == 1 || stride == 2), X3D_ERR_INVALID_ARG, "x3d_dw_wgrad: bad argument");
  const int Ho = (H + stride - 1) / stride, Wo = (W + stride - 1) / stride;
  const long orows = (long)N * T * Ho;                    // output rows; a warp walks whole rows
  const int cb = (C + 31) / 32;
  // ~8 blocks per SM in total, at least 16 rows (two per warp) each: fewer blocks = fewer atomics
  long rpb = (orows * cb + 148L * 8 - 1) / (148L * 8);
  if (rpb < 16) rpb = 16;
  rpb = (rpb + 7) / 8 * 8;
  long yb = (orows + rpb - 1) / rpb;
  if (yb > 65535) { rpb = ((orows + 65534) / 65535 + 7) / 8 * 8; yb = (orows + rpb - 1) / rpb; }
  dim3 grid(cb, (unsigned)yb);
  if (stride == 1 && C % 2 == 0 && C / 2 <= 256 && (long)N * T * H * W * C < (1L << 31) &&
      ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy)) & 7) == 0) {
    const int C2 = C / 2, bs = 256 / C2 * C2, RL = bs / C2;
    long rp = (orows + 148L * 8 - 1) / (148L * 8);         // ~8 blocks per SM in total
    if (rp < 2L * RL) rp = 2L * RL;
    rp = (rp + RL - 1) / RL * RL;
    const long nb = (orows + rp - 1) / rp;
    train::dw_wgrad_pair_kernel<<<(unsigned)nb, bs, 0, S(stream)>>>(
        reinterpret_cast<const float2*>(x), reinterpret_cast<const float2*>(dy), dwt, T, H, W, C2, pad_h, pad_w,
        (int)orows, (int)rp);
  } else if (stride == 1)
    train::dw_wgrad_kernel<1, 4><<<grid, 256, 0, S(stream)>>>(x, dy, dwt, T, H, W, Ho, Wo, C, pad_h, pad_w, orows, rpb);
  else {                                                   // measured: 2.3 ms (slide) against 3.1 ms (batched, U = 2) per step
    long rs = 16, ys = (orows + rs - 1) / rs;
    if (ys > 65535) { rs = (orows + 65534) / 65535; ys = (orows + rs - 1) / rs; }
    train::dw_wgrad_slide_kernel<<<dim3(cb, (unsigned)ys), 256, 0, S(stream)>>>(x, dy, dwt, T, H, W, Ho, Wo, C, stride, pad_h, pad_w, orows, rs);
  }
  return check_launch("x3d_dw_wgrad");
}

int x3d_stem_convs_fwd(const float* in, const float* ws, float* out, int N, int T, int H, int W, int C, void* stream) {
  X3D_REQUIRE(in && ws && out && N > 0 && T > 0 && H > 0 && W > 0 && C > 0, X3D_ERR_INVALID_ARG, "x3d_stem_convs_fwd: bad argument");
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const long rows = (long)N * T * Ho;
  X3D_REQUIRE(C % 4 == 0 && rows <= 2147483647L, X3D_ERR_UNSUPPORTED, "x3d_stem_convs_fwd: C=%d must be a multiple of 4 (and N*T*Ho < 2^31)", C);
  stem_convs_fwd_kernel<<<(unsigned)rows, 256, 0, S(stream)>>>(in, ws, out, H, W, Ho, Wo, C);
  return check_launch("x3d_stem_convs_fwd");
}

int x3d_stem_convs_wgrad(const float* in, const float* ds, double* dws, int N, int T, int H, int W, int C, void* stream) {
  X3D_REQUIRE(in && ds && dws && N > 0 && T > 0 && H > 0 && W > 0 && C > 0, X3D_ERR_INVALID_ARG, "x3d_stem_convs_wgrad: bad argument");
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const long opix = (long)N * T * Ho * Wo;
  long ppb = 1024;
  long yb = (opix + ppb - 1) / ppb;
  if (yb > 65535) { ppb = (opix + 65534) / 65535; yb = (opix + ppb - 1) / ppb; }
  if (C % 4 == 0 && C / 4 <= 64 && opix < (1L << 31) && (reinterpret_cast<uintptr_t>(ds) & 15) == 0) {
    const int C4 = C / 4, bs = 256 / C4 * C4, per = bs / C4;
    long blocks = (opix + per - 1) / per;
    if (blocks > 148L * 16) blocks = 148L * 16;
    train::stem_convs_wgrad_vec_kernel<<<(unsigned)blocks, bs, 0, S(stream)>>>(
        in, reinterpret_cast<const float4*>(ds), dws, H, W, Ho, Wo, C4, (int)opix);
    return check_launch("x3d_stem_convs_wgrad");
  }
  dim3 grid((C + 31) / 32, (unsigned)yb);
  stem_convs_wgrad_kernel<<<grid, 256, 0, S(stream)>>>(in, ds, dws, H, W, Ho, Wo, C, opix, ppb);
  return check_launch("x3d_stem_convs_wgrad");
}

int x3d_tconv_fwd(const float* in, const float* wt, float* out, int N, int T, int64_t P, int C, int kt, int flip, void* stream) {
  X3D_REQUIRE(in && wt && out && N > 0 && T > 0 && P > 0 && C > 0 && kt > 0 && kt <= 8 && (kt & 1), X3D_ERR_INVALID_ARG, "x3d_tconv_fwd: bad argument");
  X3D_REQUIRE(C % 4 == 0, X3D_ERR_UNSUPPORTED, "x3d_tconv_fwd: C=%d must be a multiple of 4", C);
  long bx = (P * (C / 4) + 255) / 256;
  if (bx > 64) bx = 64;
  X3D_REQUIRE((long)N * T * bx <= 2147483647L, X3D_ERR_UNSUPPORTED, "x3d_tconv_fwd: too many frames");
  tconv_fwd_kernel<<<(unsigned)((long)N * T * bx), 256, 0, S(stream)>>>(in, wt, out, T, P, C, kt, flip, (int)bx);
  return check_launch("x3d_tconv_fwd");
}

int x3d_tconv_wgrad(const float* s, const float* dy, double* dwt, int N, int T, int64_t P, int C, int kt, void* stream) {
  X3D_REQUIRE(s && dy && dwt && N > 0 && T > 0 && P > 0 && C > 0 && kt > 0 && kt <= 8, X3D_ERR_INVALID_ARG, "x3d_tconv_wgrad: bad argument");
  const long rows = (long)N * T * P;
  long rpb = 1024;
  long yb = (rows + rpb - 1) / rpb;
  if (yb > 65535) { rpb = (rows + 65534) / 65535; yb = (rows + rpb - 1) / rpb; }
  if (kt == 5 && C % 4 == 0 && C / 4 <= 256 &&
      ((reinterpret_cast<uintptr_t>(s) | reinterpret_cast<uintptr_t>(dy)) & 15) == 0) {
    const int C4 = C / 4, bs = 256 / C4 * C4;
    const long PC4 = P * C4, ncols = (long)N * PC4;
    long blocks = (ncols + bs - 1) / bs;
    if (blocks > 148L * 8) blocks = 148L * 8;
    tconv_wgrad_vec_kernel<5><<<(unsigned)blocks, bs, 0, S(stream)>>>(
        reinterpret_cast<const float4*>(s), reinterpret_cast<const float4*>(dy), dwt, T, PC4, C4, ncols);
    return check_launch("x3d_tconv_wgrad");
  }
  dim3 grid((C + 31) / 32, (unsigned)yb);
  tconv_wgrad_kernel<<<grid, 256, 0, S(stream)>>>(s, dy, dwt, T, P, C, kt, rows, rpb);
  return check_launch("x3d_tconv_wgrad");
}

int x3d_scale_swish_fwd(const float* y, const float* s, float* out, int64_t M, int C, int64_t rows_per_clip, void* stream) {
  X3D_REQUIRE(y && out && M > 0 && C > 0 && rows_per_clip > 0, X3D_ERR_INVALID_ARG, "x3d_scale_swish_fwd: bad argument");
  X3D_REQUIRE(C % 4 == 0 && M % rows_per_clip == 0 && M / rows_per_clip <= 65535, X3D_ERR_UNSUPPORTED,
              "x3d_scale_swish_fwd: C=%d must be a multiple of 4, M a multiple of rows_per_clip, <= 65535 clips", C);
  const long clips = M / rows_per_clip, C4 = C / 4, clip4 = rows_per_clip * C4;
  long threads = 148L * 8 * 256 / clips;                // ~8 CTAs per SM over all clips
  if (threads < 256) threads = 256;
  if (threads > clip4) threads = clip4;
  const long blocks = (threads + 255) / 256;
  long stride4 = blocks * 256 / C4 * C4;
  if (stride4 <= 0) stride4 = C4;
  dim3 grid((unsigned)blocks, (unsigned)clips);
  scale_swish_fwd_kernel<<<grid, 256, 0, S(stream)>>>(y, s, out, clip4, (int)C4, stride4);
  return check_launch("x3d_scale_swish_fwd");
}

int x3d_scale_swish_bwd(const float* dout, const float* y, const float* s, float* dy, double* ds, int64_t M, int C,
                        int64_t rows_per_clip, void* stream) {
  X3D_REQUIRE(dout && y && dy && M > 0 && C > 0 && rows_per_clip > 0 && M % rows_per_clip == 0, X3D_ERR_INVALID_ARG, "x3d_scale_swish_bwd: bad argument");
  X3D_REQUIRE((s == nullptr) == (ds == nullptr), X3D_ERR_INVALID_ARG, "x3d_scale_swish_bwd: s and ds go together");
  const long clips = M / rows_per_clip, rb = (rows_per_clip + kRowsPerBlock - 1) / kRowsPerBlock;
  X3D_REQUIRE(clips <= 65535 && rb <= 65535, X3D_ERR_UNSUPPORTED, "x3d_scale_swish_bwd: too many clips / row blocks");
  if (C % 4 == 0 && C / 4 <= 256 && clips <= 65535 &&
      ((reinterpret_cast<uintptr_t>(dout) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(dy) |
        reinterpret_cast<uintptr_t>(s)) & 15) == 0) {
    const int C4 = C / 4, bs = 256 / C4 * C4;
    const long clip4 = rows_per_clip * C4;
    long bx = (148L * 8 + clips - 1) / clips;              // ~8 CTAs per SM over all clips
    const long need = (clip4 + bs - 1) / bs;
    if (bx > need) bx = need;
    if (bx < 1) bx = 1;
    scale_swish_bwd_vec_kernel<<<dim3((unsigned)bx, (unsigned)clips), bs, 0, S(stream)>>>(
        reinterpret_cast<const float4*>(dout), reinterpret_cast<const float4*>(y), s,
        reinterpret_cast<float4*>(dy), ds, C4, clip4);
    return check_launch("x3d_scale_swish_bwd");
  }
  dim3 grid((C + 31) / 32, (unsigned)rb, (unsigned)clips);
  scale_swish_bwd_kernel<<<grid, 256, 0, S(stream)>>>(dout, y, s, dy, ds, C, rows_per_clip);
  return check_launch("x3d_scale_swish_bwd");
}

int x3d_ew(const float* a, const float* b, float* out, int64_t n, int op, void* stream) {
  X3D_REQUIRE(a && out && n > 0 && op >= 0 && op <= 5, X3D_ERR_INVALID_ARG, "x3d_ew: bad argument");
  X3D_REQUIRE(b || op == 2, X3D_ERR_INVALID_ARG, "x3d_ew: op %d needs two inputs", op);
  ew_kernel<<<ew_blocks(n), 256, 0, S(stream)>>>(a, b, out, n, op);
  return check_launch("x3d_ew");
}

int x3d_pool_bwd(const float* dm, float* dy, int64_t M, int C, int64_t rows_per_clip, float scale, int accumulate, void* stream) {
  X3D_REQUIRE(dm && dy && M > 0 && C > 0 && rows_per_clip > 0, X3D_ERR_INVALID_ARG, "x3d_pool_bwd: bad argument");
  pool_bwd_kernel<<<ew_blocks(M * C), 256, 0, S(stream)>>>(dm, dy, M * C, C, rows_per_clip, scale, accumulate);
  return check_launch("x3d_pool_bwd");
}

int x3d_strided_add(const float* src, float* dst, int NT, int Ho, int Wo, int Hi, int Wi, int stride, int C, void* stream) {
  X3D_REQUIRE(src && dst && NT > 0 && Ho > 0 && Wo > 0 && C > 0 && stride >= 1, X3D_ERR_INVALID_ARG, "x3d_strided_add: bad argument");
  const long total = (long)NT * Ho * Wo * C;
  strided_add_kernel<<<ew_blocks(total), 256, 0, S(stream)>>>(src, dst, Ho, Wo, Hi, Wi, stride, C, total);
  return check_launch("x3d_strided_add");
}

int x3d_dropout_mask(float* mask, int64_t n, float rate, uint64_t seed, void* stream) {
  X3D_REQUIRE(mask && n > 0 && rate >= 0.f && rate < 1.f, X3D_ERR_INVALID_ARG, "x3d_dropout_mask: bad argument");
  dropout_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, S(stream)>>>(mask, n, rate, seed);
  return check_launch("x3d_dropout_mask");
}

int x3d_softmax_xent(const float* logits, const int32_t* labels, float* loss, float* dlogits, int N, int ncls,
                     float gscale, void* stream) {
  X3D_REQUIRE(logits && labels && loss && dlogits && N > 0 && ncls > 0, X3D_ERR_INVALID_ARG, "x3d_softmax_xent: bad argument");
  softmax_xent_kernel<<<N, 256, 0, S(stream)>>>(logits, labels, loss, dlogits, ncls, gscale);
  return check_launch("x3d_softmax_xent");
}

int x3d_adam_step(float* w, const float* grad, float* m, float* v, const float* wd, int64_t n, float lr_t,
                  float beta1, float beta2, float eps, void* stream) {
  X3D_REQUIRE(w && grad && m && v && wd && n > 0, X3D_ERR_INVALID_ARG, "x3d_adam_step: bad argument");
  adam_kernel<<<ew_blocks(n), 256, 0, S(stream)>>>(w, grad, m, v, wd, n, lr_t, beta1, beta2, eps);
  return check_launch("x3d_adam_step");
}

int x3d_sgd_nesterov_step(float* w, const float* grad, float* v, const float* wd, int64_t n, float lr, float momentum,
                          void* stream) {
  X3D_REQUIRE(w && grad && v && wd && n > 0, X3D_ERR_INVALID_ARG, "x3d_sgd_nesterov_step: bad argument");
  sgd_nesterov_kernel<<<ew_blocks(n), 256, 0, S(stream)>>>(w, grad, v, wd, n, lr, momentum);
  return check_launch("x3d_sgd_nesterov_step");
}

}  // extern "C"
