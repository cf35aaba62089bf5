// fp32 pointwise (1x1x1) convolution on the Blackwell tensor cores with the 3xTF32 split:
//   D[M, Nc] = act(bias + A[M, K] * B[Nc, K]^T),   fp32 in, fp32 out, fp32-level accuracy.
// Every fp32 operand x is written as hi + lo with hi = x rounded to TF32 (10 mantissa bits) and
// lo = x - hi (exact in fp32); the product is accumulated as A_lo*B_hi + A_hi*B_lo + A_hi*B_hi by
// three tcgen05.mma.kind::tf32 per K step into one fp32 TMEM accumulator (the lo*lo term, 2^-22 of
// the product, is dropped).  This is the training path's GEMM (the reference trains in fp32,
// train.py:85-152): forward of Bottleneck.a / c, the shortcut, conv5, fc1, fc2 (model.py:246-253,
// 292-299, 360-367, 78-108) with B = W^T, and backward-data of the same layers with B = W.
//
//   * B arrives pre-split from x3d_tf32_split: two fp32 planes [2][Nc][K] (reduction dim contiguous);
//   * per (M tile, 32-column K chunk) the producer lane TMA-loads A[128 x 32] fp32 and the chunk of
//     both B planes (128B swizzle; rows / columns outside the tensors are zero-filled);
//   * 8 transform warps split the landed A tile in shared memory: hi in place, lo into a second
//     buffer at the same swizzled offsets;
//   * one elected thread issues the MMAs (M=128, N=NT<=256, K=8) into a double-buffered TMEM
//     accumulator; tcgen05.commit frees ring stages / publishes the accumulator;
//   * 4 epilogue warps drain TMEM (tcgen05.ld), add the bias, apply ReLU and store fp32 rows through
//     128B-swizzled staging and TMA box stores (clipped at M / Nc).
// The same pipeline has a bf16 operand mode for the mixed-precision training step
// (x3d_pw_bf16_train_fwd, see pw_tc_body): bf16 RNE operands, one kind::f16 MMA per K=16 step.
#include <stdlib.h>

#include "tma_common.cuh"

namespace x3d {
namespace tf32tc {

using namespace ptx;

constexpr int kBlockM = 128, kBlockK = 32;              // 32 fp32 = one 128-byte swizzle row
constexpr int kATile = kBlockM * kBlockK * 4;           // 16 KiB
constexpr int kEpiWarps = 4, kXfWarps = 8;
constexpr int kThreads = 64 + 32 * (kEpiWarps + kXfWarps);

__device__ __forceinline__ void tcgen05_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// K-major operand, 128-byte swizzle, 8-row atoms stacked every 1024 B (as in x3d_pw_tc.cu).
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor: D = f32, A = B = TF32 (format code 2), both K-major, M = 128, N = n.
__device__ __forceinline__ uint32_t make_idesc_tf32(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(kBlockM >> 4) << 24);
}
// The same for kind::f16 with A = B = BF16 (format code 1).
__device__ __forceinline__ uint32_t make_idesc_bf16(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(kBlockM >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_s(uint32_t dst, const CUtensorMap* map, int c0, int c1,
                                              uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// hi = x rounded to nearest TF32 (ties away: add half an ulp of the 13 dropped bits, clear them),
// lo = x - hi, exact.  Integer ops only: cvt.rna.tf32 would run on the 16-lane conversion pipe.
__device__ __forceinline__ void split_tf32(uint32_t x, uint32_t& hi, uint32_t& lo) {
  hi = (x + 0x1000u) & 0xffffe000u;
  lo = __float_as_uint(__uint_as_float(x) - __uint_as_float(hi));
}

// {lo, hi} -> one bf16x2 word (lo in the low half, the lower address), round-to-nearest-even as
// torch's .to(torch.bfloat16)
__device__ __forceinline__ uint32_t pack_bf16x2_rn(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}

struct Params {
  const float* bias;
  double* stats;   // [2][Nc] column sums / sums of squares of D (BatchNorm batch statistics), or nullptr
  long M;
  int Nc;          // output columns
  int NT;          // N tile (multiple of 32, <= 256)
  int KC;          // 32-wide K chunks (bf16: 64-wide)
  int k8_last;     // K=8 (bf16: K=16) MMA steps in the last chunk (1..4)
  int stages;      // ring depth
  int stage_bytes; // 2 * kATile + 2 * NT * 128 (bf16: 3 * kATile + NT * 128)
  int tmem_cols;   // power of two >= 2 * NT
  int relu;
};

// kBf16 = false: the 3xTF32 split above.  kBf16 = true: the bf16 operand mode of the mixed-precision
// training step.  A ring stage then holds two fp32 A boxes (K columns [64kc, 64kc+32) and [+32, +64)),
// the bf16 RNE tile of both (128 rows x 64 bf16 = one 128-byte swizzle row each, the layout
// tcgen05.mma kind::f16 reads) and one bf16 B chunk [NT][64] (tmB 2-D over the bf16 [Nc][K] weights);
// one MMA per K=16 step.  The epilogue is the same.
template <bool kBf16>
__device__ __forceinline__ void pw_tc_body(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmD,
                                           const Params p) {
  extern __shared__ __align__(1024) uint8_t tf_smem_raw[];
  const uint32_t raw_s = smem_u32(tf_smem_raw);
  const uint32_t base_s = (raw_s + 1023u) & ~1023u;
  uint8_t* smem = tf_smem_raw + (base_s - raw_s);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.y * p.NT;
  const int b_plane = p.NT * 128;                          // bytes of one B plane chunk

  // layout: [stages] x {A_hi, A_lo, B_hi, B_lo} | output staging 2 x 16 KiB | bias | barriers
  const uint32_t ring_s = base_s;
  const uint32_t out_s = ring_s + p.stages * p.stage_bytes;
  float* sBias = reinterpret_cast<float*>(smem + p.stages * p.stage_bytes + 2 * kATile);
  uint64_t* bars = reinterpret_cast<uint64_t*>(sBias + 256);
  uint64_t* full = bars;                      // [stages]  TMA landed
  uint64_t* empty = full + p.stages;          // [stages]  MMAs done reading
  uint64_t* xform = empty + p.stages;         // [stages]  A split written
  uint64_t* t_full = xform + p.stages;        // [2] accumulator ready
  uint64_t* t_empty = t_full + 2;             // [2] accumulator drained
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);

  for (int i = threadIdx.x; i < p.NT; i += blockDim.x) {
    const int col = n0 + i;
    sBias[i] = (p.bias != nullptr && col < p.Nc) ? p.bias[col] : 0.f;
  }
  if (warp == 0 && elect_one()) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    prefetch_tmap(&tmD);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
      mbar_init(&xform[s], 32 * kXfWarps);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&t_full[i], 1);
      mbar_init(&t_empty[i], 32 * kEpiWarps);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(tmem_slot)),
                 "r"(static_cast<uint32_t>(p.tmem_cols))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_before_sync();
  __syncthreads();
  tcgen05_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const long num_tiles = (p.M + kBlockM - 1) / kBlockM;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      int s = 0;
      uint32_t ph = 0;
      for (long tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int row0 = static_cast<int>(tile * kBlockM);
        for (int kc = 0; kc < p.KC; ++kc) {
          mbar_wait(&empty[s], ph ^ 1);
          const uint32_t st = ring_s + s * p.stage_bytes;
          if constexpr (kBf16) {
            // both A boxes always: a box past K is zero-filled and still counts its bytes
            mbar_expect_tx(&full[s], static_cast<uint32_t>(2 * kATile + b_plane));
            tma_load_2d_s(st, &tmA, kc * 2 * kBlockK, row0, &full[s]);
            tma_load_2d_s(st + kATile, &tmA, kc * 2 * kBlockK + kBlockK, row0, &full[s]);
            tma_load_2d_s(st + 3 * kATile, &tmB, kc * 2 * kBlockK, n0, &full[s]);
          } else {
            mbar_expect_tx(&full[s], static_cast<uint32_t>(kATile + 2 * b_plane));
            tma_load_2d_s(st, &tmA, kc * kBlockK, row0, &full[s]);
            tma_load_3d(st + 2 * kATile, &tmB, kc * kBlockK, n0, 0, &full[s]);
            tma_load_3d(st + 2 * kATile + b_plane, &tmB, kc * kBlockK, n0, 1, &full[s]);
          }
          if (++s == p.stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    const uint32_t idesc = kBf16 ? make_idesc_bf16(p.NT) : make_idesc_tf32(p.NT);
    int s = 0;
    uint32_t ph = 0;
    long it = 0;
    for (long tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int as = static_cast<int>(it & 1);
      const uint32_t aph = static_cast<uint32_t>((it >> 1) & 1);
      mbar_wait(&t_empty[as], aph ^ 1);
      tcgen05_after_sync();
      const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * p.NT);
      for (int kc = 0; kc < p.KC; ++kc) {
        mbar_wait(&xform[s], ph);
        tcgen05_after_sync();
        if constexpr (kBf16) {
          if (elect_one()) {
            const uint32_t a_bf = ring_s + s * p.stage_bytes + 2 * kATile, b_bf = a_bf + kATile;
            const int nk = (kc == p.KC - 1) ? p.k8_last : 4;
            for (int k = 0; k < nk; ++k) {
              const uint32_t o = k * 32;                       // 16 bf16 = 32 bytes per K step
              umma_f16(d_tmem, make_desc_sw128(a_bf + o), make_desc_sw128(b_bf + o), idesc, (kc | k) != 0 ? 1u : 0u);
            }
            umma_commit(&empty[s]);
            if (kc == p.KC - 1) umma_commit(&t_full[as]);
          }
        } else if (elect_one()) {
          const uint32_t a_hi = ring_s + s * p.stage_bytes, a_lo = a_hi + kATile;
          const uint32_t b_hi = a_hi + 2 * kATile, b_lo = b_hi + b_plane;
          const int nk = (kc == p.KC - 1) ? p.k8_last : 4;
          for (int k = 0; k < nk; ++k) {
            const uint32_t o = k * 32;                       // 8 fp32 = 32 bytes per K step
            // small terms first, the dominant product last
            umma_tf32(d_tmem, make_desc_sw128(a_lo + o), make_desc_sw128(b_hi + o), idesc, (kc | k) != 0 ? 1u : 0u);
            umma_tf32(d_tmem, make_desc_sw128(a_hi + o), make_desc_sw128(b_lo + o), idesc, 1u);
            umma_tf32(d_tmem, make_desc_sw128(a_hi + o), make_desc_sw128(b_hi + o), idesc, 1u);
          }
          umma_commit(&empty[s]);
          if (kc == p.KC - 1) umma_commit(&t_full[as]);
        }
        __syncwarp();
        if (++s == p.stages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp < 2 + kEpiWarps) {
    // ------------------------------------------------------------------ epilogue (4 warps)
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    const bool leader = warp == 2 && lane == 0;
    const int r_loc = q * 32 + lane;
    const uint32_t sw_row = static_cast<uint32_t>(r_loc) * 128, sw_x = static_cast<uint32_t>(r_loc & 7);
    const int n_sub = (p.NT + 31) >> 5;           // 32-column (128-byte) output boxes
    const uint32_t bias_s = smem_u32(sBias);
    uint32_t sub_ctr = 0;
    long it = 0;
    // running column sums / sums of squares of this thread's (column, 32-row group) over all tiles of the
    // CTA: one pair of global atomics per column and CTA at the end, not per tile (12.5 k tiles hitting
    // the same 56 addresses measured +4 ms per step)
    double acc1[8], acc2[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc1[i] = acc2[i] = 0.0;
    for (long tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int as = static_cast<int>(it & 1);
      const uint32_t aph = static_cast<uint32_t>((it >> 1) & 1);
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(as * p.NT);
      mbar_wait(&t_full[as], aph);
      tcgen05_after_sync();
#pragma unroll
      for (int sb = 0; sb < 8; ++sb) {
        if (sb >= n_sub || n0 + sb * 32 >= p.Nc) break;          // uniform across the CTA
        const uint32_t buf = out_s + (sub_ctr & 1) * kATile + sw_row;
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          const int c0 = sb * 32 + g * 16;
          uint32_t v[16];
          tmem_ld16(taddr + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int h = 0; h < 4; ++h) {
            float4 b;
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "r"(bias_s + (c0 + h * 4) * 4));
            float y0 = __uint_as_float(v[h * 4 + 0]) + b.x, y1 = __uint_as_float(v[h * 4 + 1]) + b.y;
            float y2 = __uint_as_float(v[h * 4 + 2]) + b.z, y3 = __uint_as_float(v[h * 4 + 3]) + b.w;
            if (p.relu) { y0 = fmaxf(y0, 0.f); y1 = fmaxf(y1, 0.f); y2 = fmaxf(y2, 0.f); y3 = fmaxf(y3, 0.f); }
            const uint32_t chunk = static_cast<uint32_t>(g * 4 + h);            // 16-byte chunk 0..7
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(buf + ((chunk ^ sw_x) << 4)),
                         "f"(y0), "f"(y1), "f"(y2), "f"(y3) : "memory");
          }
        }
        if (sb == n_sub - 1 || n0 + (sb + 1) * 32 >= p.Nc) {
          tcgen05_before_sync();                  // last TMEM read of this tile is done
          mbar_arrive(&t_empty[as]);
        }
        fence_proxy_async();
        // every store issued so far has finished reading its staging buffer (checked here, after this
        // box is written): once the barrier is passed the OTHER buffer is free for the next box
        if (leader) tma_store_wait_read<0>();
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (leader) {
          tma_store_2d(&tmD, out_s + (sub_ctr & 1) * kATile, n0 + sb * 32, static_cast<int>(tile * kBlockM));
          tma_store_commit();
        }
        if (p.stats != nullptr) {
          // BatchNorm statistics of the layer this GEMM feeds (model.py:254,300,89 in training mode),
          // taken from the staged tile while the TMA store reads it: thread = (column, 32-row group);
          // rows past M are exact zeros (zero-filled A rows, no bias), so they add nothing
          const int c = lane, rg = warp - 2;
          const uint32_t cbase = out_s + (sub_ctr & 1) * kATile + static_cast<uint32_t>(c & 3) * 4;
          float s1 = 0.f, s2 = 0.f;
#pragma unroll 8
          for (int i = 0; i < 32; ++i) {
            const int r = rg * 32 + i;
            float v;
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(cbase + r * 128 + ((static_cast<uint32_t>(c >> 2) ^ static_cast<uint32_t>(r & 7)) << 4)));
            s1 += v;
            s2 = fmaf(v, v, s2);
          }
          acc1[sb] += static_cast<double>(s1);
          acc2[sb] += static_cast<double>(s2);
        }
        ++sub_ctr;
      }
    }
    if (leader) tma_store_wait_read<0>();
    if (p.stats != nullptr) {
#pragma unroll
      for (int sb = 0; sb < 8; ++sb) {
        const int col = n0 + sb * 32 + lane;
        if (sb < n_sub && col < p.Nc) {
          atomicAdd(p.stats + col, acc1[sb]);
          atomicAdd(p.stats + p.Nc + col, acc2[sb]);
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ transform: A -> (hi, lo)
    const int tt = threadIdx.x - (64 + 32 * kEpiWarps);        // 0..255
    int s = 0;
    uint32_t ph = 0;
    for (long tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      for (int kc = 0; kc < p.KC; ++kc) {
        mbar_wait(&full[s], ph);
        if constexpr (kBf16) {
          // 16-byte bf16 chunk e = (row r, K columns 8c..8c+8) from the fp32 chunks 2(c%4), 2(c%4)+1 of box c/4
          const uint32_t st = ring_s + s * p.stage_bytes;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int e = tt + i * 256, r = e >> 3, c = e & 7;
            const uint32_t x = static_cast<uint32_t>(r & 7), row = st + static_cast<uint32_t>(r) * 128;
            const uint32_t src = row + (c >> 2) * kATile, c0 = static_cast<uint32_t>((c & 3) * 2);
            float f[8];
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(f[0]), "=f"(f[1]), "=f"(f[2]), "=f"(f[3]) : "r"(src + ((c0 ^ x) << 4)));
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(f[4]), "=f"(f[5]), "=f"(f[6]), "=f"(f[7]) : "r"(src + (((c0 + 1) ^ x) << 4)));
            uint32_t b[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = pack_bf16x2_rn(f[2 * j], f[2 * j + 1]);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(row + 2 * kATile + ((static_cast<uint32_t>(c) ^ x) << 4)),
                         "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]) : "memory");
          }
          fence_proxy_async();
          mbar_arrive(&xform[s]);
          if (++s == p.stages) { s = 0; ph ^= 1; }
          continue;
        }
        const uint32_t a_hi = ring_s + s * p.stage_bytes + tt * 16;      // 16-byte vectors, any order: the
#pragma unroll                                                           // split is element-wise
        for (int i = 0; i < 4; ++i) {
          const uint32_t addr = a_hi + i * (256 * 16);
          uint32_t x[4], hi[4], lo[4];
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(x[0]), "=r"(x[1]), "=r"(x[2]), "=r"(x[3]) : "r"(addr));
#pragma unroll
          for (int j = 0; j < 4; ++j) split_tf32(x[j], hi[j], lo[j]);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(hi[0]), "r"(hi[1]), "r"(hi[2]), "r"(hi[3]) : "memory");
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr + kATile), "r"(lo[0]), "r"(lo[1]), "r"(lo[2]), "r"(lo[3]) : "memory");
        }
        fence_proxy_async();
        mbar_arrive(&xform[s]);
        if (++s == p.stages) { s = 0; ph ^= 1; }
      }
    }
  }

  tcgen05_before_sync();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"(static_cast<uint32_t>(p.tmem_cols))
                 : "memory");
  }
}

__global__ void __launch_bounds__(kThreads, 1)
pw_tf32_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const __grid_constant__ CUtensorMap tmD, const Params p) {
  pw_tc_body<false>(tmA, tmB, tmD, p);
}

__global__ void __launch_bounds__(kThreads, 1)
pw_bf16_train_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                        const __grid_constant__ CUtensorMap tmD, const Params p) {
  pw_tc_body<true>(tmA, tmB, tmD, p);
}

// out[0][r][c] = hi(x), out[1][r][c] = lo(x) with x = transpose ? W[c][r] : W[r][c]
__global__ void tf32_split_kernel(const float* __restrict__ W, float* __restrict__ out, int rows, int cols, int ld,
                                  int transpose) {
  const long n = static_cast<long>(rows) * cols;
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / cols), c = static_cast<int>(i - static_cast<long>(r) * cols);
    const float x = transpose ? W[static_cast<long>(c) * ld + r] : W[static_cast<long>(r) * ld + c];
    uint32_t hi, lo;
    split_tf32(__float_as_uint(x), hi, lo);
    out[i] = __uint_as_float(hi);
    out[n + i] = __uint_as_float(lo);
  }
}

// x3d_bf16_round: out[r][c] = bf16_rn(transpose ? W[c][r] : W[r][c]), rows of pitch round_up(cols, 8),
// the padding columns zero (TMA needs 16-byte row strides).
__global__ void bf16_round_kernel(const float* __restrict__ W, uint16_t* __restrict__ out, int rows, int cols,
                                  int pitch, int ld, int transpose) {
  const long n = static_cast<long>(rows) * pitch;
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / pitch), c = static_cast<int>(i - static_cast<long>(r) * pitch);
    float x = 0.f;
    if (c < cols) x = transpose ? W[static_cast<long>(c) * ld + r] : W[static_cast<long>(r) * ld + c];
    out[i] = static_cast<uint16_t>(pack_bf16x2_rn(x, 0.f) & 0xffffu);
  }
}

}  // namespace tf32tc
}  // namespace x3d

using namespace x3d;

extern "C" int x3d_tf32_split(const float* W, float* out, int rows, int cols, int ld, int transpose, void* stream) {
  X3D_REQUIRE(W && out && rows > 0 && cols > 0 && ld > 0, X3D_ERR_INVALID_ARG, "x3d_tf32_split: bad argument");
  const long n = (long)rows * cols;
  long blocks = (n + 255) / 256;
  if (blocks > 1184) blocks = 1184;
  tf32tc::tf32_split_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(W, out, rows, cols, ld, transpose);
  return check_launch("x3d_tf32_split");
}

extern "C" int x3d_bf16_round(const float* W, void* out, int rows, int cols, int ld, int transpose, void* stream) {
  X3D_REQUIRE(W && out && rows > 0 && cols > 0 && ld > 0, X3D_ERR_INVALID_ARG, "x3d_bf16_round: bad argument");
  X3D_REQUIRE(ld >= (transpose ? rows : cols), X3D_ERR_INVALID_ARG, "x3d_bf16_round: ld=%d too small", ld);
  const int pitch = (cols + 7) / 8 * 8;
  const long n = (long)rows * pitch;
  long blocks = (n + 255) / 256;
  if (blocks > 1184) blocks = 1184;
  tf32tc::bf16_round_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      W, static_cast<uint16_t*>(out), rows, cols, pitch, ld, transpose);
  return check_launch("x3d_bf16_round");
}

// Shared host side of both operand modes.  bf16: B is bf16 [Nc][round_up(K, 8)] from x3d_bf16_round;
// otherwise the two fp32 planes [2][Nc][K] of x3d_tf32_split.
static int pw_tc_launch(const char* fn, bool bf16, const float* A, const void* B, const float* bias, float* D,
                        int64_t M, int K, int Nc, int lda, int ldd, int relu, double* stats, void* stream) {
  X3D_REQUIRE(A && B && D, X3D_ERR_INVALID_ARG, "%s: null pointer", fn);
  X3D_REQUIRE(!stats || (!bias && !relu), X3D_ERR_INVALID_ARG,
              "%s: column statistics are those of the plain product (no bias, no ReLU)", fn);
  X3D_REQUIRE(M > 0 && M < (1L << 31), X3D_ERR_INVALID_ARG, "%s: M out of range", fn);
  X3D_REQUIRE(K > 0 && K % 4 == 0 && lda % 4 == 0 && lda >= K, X3D_ERR_INVALID_ARG,
              "%s: K=%d / lda=%d must be multiples of 4", fn, K, lda);
  X3D_REQUIRE(Nc > 0 && Nc % 4 == 0 && ldd % 4 == 0 && ldd >= Nc, X3D_ERR_INVALID_ARG,
              "%s: Nc=%d / ldd=%d must be multiples of 4", fn, Nc, ldd);
  X3D_REQUIRE((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(B) & 15) == 0 &&
              (reinterpret_cast<uintptr_t>(D) & 15) == 0, X3D_ERR_INVALID_ARG, "%s: pointers must be 16-byte aligned", fn);
  X3D_REQUIRE(device_sm_count() > 0 && device_is_sm100(), X3D_ERR_NO_DEVICE, "%s: needs an sm_100 device", fn);
  EncodeTiledFn enc = tensor_map_encoder();
  X3D_REQUIRE(enc != nullptr, X3D_ERR_NO_DEVICE, "%s: cuTensorMapEncodeTiled unavailable", fn);

  // N tiling: one tile up to 256 columns, else the fewest tiles of a multiple of 32 columns
  int n_tiles = (Nc + 255) / 256;
  int NT = ((Nc + n_tiles - 1) / n_tiles + 31) / 32 * 32;
  n_tiles = (Nc + NT - 1) / NT;
  const int kchunk = bf16 ? 2 * tf32tc::kBlockK : tf32tc::kBlockK, kstep = bf16 ? 16 : 8;
  const int KC = (K + kchunk - 1) / kchunk;
  const int k8_last = ((K - (KC - 1) * kchunk) + kstep - 1) / kstep;
  const int stage_bytes = bf16 ? 3 * tf32tc::kATile + NT * 128 : 2 * tf32tc::kATile + 2 * NT * 128;
  const int fixed = 1024 /*align*/ + 2 * tf32tc::kATile /*staging*/ + 1024 /*bias*/ + 512 /*barriers*/;
  int stages = (device_max_smem() - fixed) / stage_bytes;
  X3D_REQUIRE(stages >= 2, X3D_ERR_UNSUPPORTED, "%s: NT=%d does not fit two ring stages", fn, NT);
  if (stages > 4) stages = 4;
  int tmem_cols = 32;
  while (tmem_cols < 2 * NT) tmem_cols *= 2;
  X3D_REQUIRE(tmem_cols <= 512, X3D_ERR_UNSUPPORTED, "%s: NT=%d needs too much TMEM", fn, NT);

  CUtensorMap tmA, tmB, tmD;
  cuuint32_t estr[3] = {1, 1, 1};
  {
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)M};
    cuuint64_t strides[1] = {(cuuint64_t)lda * 4};
    cuuint32_t box[2] = {32, 128};
    CUresult r = enc(&tmA, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(A), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    X3D_REQUIRE(r == CUDA_SUCCESS, X3D_ERR_LAUNCH, "%s: tensor map for A failed (%d; K=%d M=%ld lda=%d)", fn, (int)r, K, (long)M, lda);
  }
  if (bf16) {
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)Nc};
    cuuint64_t strides[1] = {(cuuint64_t)((K + 7) / 8 * 8) * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)NT};
    CUresult r = enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(B), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    X3D_REQUIRE(r == CUDA_SUCCESS, X3D_ERR_LAUNCH, "%s: tensor map for B failed (%d; K=%d Nc=%d NT=%d)", fn, (int)r, K, Nc, NT);
  } else {
    cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)Nc, 2};
    cuuint64_t strides[2] = {(cuuint64_t)K * 4, (cuuint64_t)K * 4 * (cuuint64_t)Nc};
    cuuint32_t box[3] = {32, (cuuint32_t)NT, 1};
    CUresult r = enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(B), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    X3D_REQUIRE(r == CUDA_SUCCESS, X3D_ERR_LAUNCH, "%s: tensor map for B failed (%d; K=%d Nc=%d NT=%d)", fn, (int)r, K, Nc, NT);
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)Nc, (cuuint64_t)M};
    cuuint64_t strides[1] = {(cuuint64_t)ldd * 4};
    cuuint32_t box[2] = {32, 128};
    CUresult r = enc(&tmD, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, D, dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    X3D_REQUIRE(r == CUDA_SUCCESS, X3D_ERR_LAUNCH, "%s: tensor map for D failed (%d; Nc=%d M=%ld ldd=%d)", fn, (int)r, Nc, (long)M, ldd);
  }
  tf32tc::Params p;
  p.bias = bias; p.stats = stats; p.M = M; p.Nc = Nc; p.NT = NT; p.KC = KC; p.k8_last = k8_last; p.stages = stages;
  p.stage_bytes = stage_bytes; p.tmem_cols = tmem_cols; p.relu = relu;
  const size_t smem = (size_t)fixed + (size_t)stages * stage_bytes;
  const long num_tiles = (M + tf32tc::kBlockM - 1) / tf32tc::kBlockM;
  int gx = device_sm_count() / n_tiles;
  if (gx < 1) gx = 1;
  if (gx > num_tiles) gx = (int)num_tiles;
  dim3 grid(gx, n_tiles);
  static SmemOptIn optin_tf32, optin_bf16;
  const cudaError_t e = bf16 ? ensure_dynamic_smem(tf32tc::pw_bf16_train_tc_kernel, optin_bf16, smem, false)
                             : ensure_dynamic_smem(tf32tc::pw_tf32_tc_kernel, optin_tf32, smem, false);
  X3D_REQUIRE(e == cudaSuccess, X3D_ERR_LAUNCH, "%s: smem attribute: %s", fn, cudaGetErrorString(e));
  if (bf16)
    tf32tc::pw_bf16_train_tc_kernel<<<grid, tf32tc::kThreads, smem, static_cast<cudaStream_t>(stream)>>>(tmA, tmB, tmD, p);
  else
    tf32tc::pw_tf32_tc_kernel<<<grid, tf32tc::kThreads, smem, static_cast<cudaStream_t>(stream)>>>(tmA, tmB, tmD, p);
  return check_launch(fn);
}

extern "C" int x3d_pw_tf32_fwd(const float* A, const float* Bsplit, const float* bias, float* D, int64_t M, int K,
                               int Nc, int lda, int ldd, int relu, double* stats, void* stream) {
  return pw_tc_launch("x3d_pw_tf32_fwd", false, A, Bsplit, bias, D, M, K, Nc, lda, ldd, relu, stats, stream);
}

extern "C" int x3d_pw_bf16_train_fwd(const float* A, const void* Wb, const float* bias, float* D, int64_t M, int K,
                                     int Nc, int lda, int ldd, int relu, double* stats, void* stream) {
  return pw_tc_launch("x3d_pw_bf16_train_fwd", true, A, Wb, bias, D, M, K, Nc, lda, ldd, relu, stats, stream);
}
