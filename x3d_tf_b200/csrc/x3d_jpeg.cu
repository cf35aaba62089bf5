// Baseline JPEG decoding of TFRecord video frames (the reference's tf.io.decode_jpeg in
// dataloader.py:66-91, 150-174), in three stages that reproduce libjpeg-turbo's decompressor in its
// default libjpeg-6b mode bit for bit (pure integer arithmetic):
//   x3d_jpeg_entropy  Huffman decoding (jdhuff.c)                  -> int16 coefficient blocks
//   x3d_jpeg_entropy_rst  the same for frames with restart intervals, one thread per interval
//   x3d_jpeg_idct     dequantisation + jidctint.c / jidctfst.c     -> per-component sample planes
//   x3d_jpeg_color    jdsample.c h2v2 / h2v1_fancy_upsample + jdcolor.c -> packed [H][W][3] RGB frames
// Layouts and preconditions: include/x3d_b200.h.
#include "common.cuh"

namespace x3d {
namespace jpeg {

__constant__ uint8_t kNatural[64] = {
    0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
    41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
    30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// jddctmgr.c aanscales (natural order, scaled by 2^14), for the IFAST multiplier table
__constant__ int16_t kAanScales[64] = {
    16384, 22725, 21407, 19266, 16384, 12873, 8867,  4520,  22725, 31521, 29692, 26722, 22725,
    17855, 12299, 6270,  21407, 29692, 27969, 25172, 21407, 16819, 11585, 5906,  19266, 26722,
    25172, 22654, 19266, 15137, 10426, 5315,  16384, 22725, 21407, 19266, 16384, 12873, 8867,
    4520,  12873, 17855, 16819, 15137, 12873, 10114, 6967,  3552,  8867,  12299, 11585, 10426,
    8867,  6967,  4799,  2446,  4520,  6270,  5906,  5315,  4520,  3552,  2446,  1247};

// ---------------------------------------------------------------------------------------------
// Stage 1: entropy decoding, one warp per frame.
//
// The unstuffed entropy-coded bytes pass through a per-warp ring in shared memory.  All 32 lanes
// refill it a chunk at a time (coalesced byte loads, FF 00 -> FF by a ballot / prefix count), and
// they keep at least kAhead bytes ahead of lane 0's read position, more than one MCU can need (6
// blocks of at most 16 + 11 + 63 * (16 + 10) bits = 1250 bytes).  Lane 0 decodes one MCU at a time
// into zeroed blocks in shared memory; the warp then flushes each block with 16-byte stores (one
// 128-byte line per block).  Past the segment's end lane 0 reads zeros, as libjpeg does, and the
// frame is flagged if the decode consumes any of them.
constexpr int kRing = 4096;                // ring bytes (power of two)
constexpr int kChunk = 1024;               // input bytes per refill
constexpr int kAhead = 2048;               // refill while fewer unread bytes are staged
constexpr int kMaxBlocks = 6;              // blocks per MCU (4:2:0)

struct HuffSmem {
  uint16_t lookup[4][256];                 // dc0, dc1, ac0, ac1
  int32_t maxcode[4][18];
  int32_t valoffset[4][18];
  uint8_t huffval[4][256];
};

struct EntropySmem {
  HuffSmem h;
  uint8_t ring[kRing];
  int16_t blk[kMaxBlocks][64];
};

struct BitReader {
  uint64_t acc;        // MSB-aligned
  int nbits;
  int64_t rpos;        // unstuffed bytes pulled into acc
  const uint8_t* ring;

  __device__ __forceinline__ void fill(int64_t staged) {
    while (nbits <= 56) {
      const uint64_t b = rpos < staged ? ring[rpos & (kRing - 1)] : 0u;   // zeros past the end
      acc |= b << (56 - nbits);
      nbits += 8;
      ++rpos;
    }
  }
  __device__ __forceinline__ uint32_t peek(int n) const { return static_cast<uint32_t>(acc >> (64 - n)); }
  __device__ __forceinline__ void skip(int n) { acc <<= n; nbits -= n; }
};

// jdhuff.c HUFF_DECODE / jpeg_huff_decode: returns the symbol, or -1 for a bad code
__device__ __forceinline__ int huff_decode(BitReader& br, int64_t staged, const HuffSmem& h, int t) {
  br.fill(staged);
  const uint32_t look = h.lookup[t][br.peek(8)];
  int l = look >> 8;
  if (l <= 8) {
    br.skip(l);
    return look & 0xff;
  }
  // slow path: codes longer than 8 bits (acc holds >= 57 bits, enough for 16)
  int32_t code = static_cast<int32_t>(br.peek(9));
  l = 9;
  while (l <= 16 && code > h.maxcode[t][l]) {
    ++l;
    code = static_cast<int32_t>(br.peek(l));
  }
  if (l > 16) return -1;
  br.skip(l);
  return h.huffval[t][(code + h.valoffset[t][l]) & 0xff];
}

__device__ __forceinline__ int get_bits(BitReader& br, int64_t staged, int s) {
  br.fill(staged);
  const int r = static_cast<int>(br.peek(s));
  br.skip(s);
  return r;
}

__device__ __forceinline__ int huff_extend(int r, int s) {
  return r < (1 << (s - 1)) ? r + static_cast<int>((~0u << s) + 1u) : r;
}

__global__ void __launch_bounds__(32)
entropy_kernel(const uint8_t* __restrict__ data, const x3d_jpeg_frame* __restrict__ frames,
               const x3d_jpeg_tables* __restrict__ tables, int16_t* __restrict__ coef,
               int32_t* __restrict__ status) {
  __shared__ __align__(16) EntropySmem sm;
  const int lane = threadIdx.x;
  const x3d_jpeg_frame fr = frames[blockIdx.x];
  const x3d_jpeg_tables* tb = tables + fr.tables;

  // Huffman tables of this frame's header
  for (int i = lane; i < 4 * 256; i += 32) {
    const int t = i >> 8, k = i & 255;
    const x3d_jpeg_huff& src = t < 2 ? tb->dc[t] : tb->ac[t - 2];
    sm.h.lookup[t][k] = src.lookup[k];
    sm.h.huffval[t][k] = src.huffval[k];
  }
  for (int i = lane; i < 4 * 18; i += 32) {
    const int t = i / 18, k = i - t * 18;
    const x3d_jpeg_huff& src = t < 2 ? tb->dc[t] : tb->ac[t - 2];
    sm.h.maxcode[t][k] = src.maxcode[k];
    sm.h.valoffset[t][k] = src.valoffset[k];
  }
  for (int i = lane; i < kMaxBlocks * 64 / 8; i += 32) reinterpret_cast<int4*>(&sm.blk[0][0])[i] = make_int4(0, 0, 0, 0);

  const int hs = fr.hs, vs = fr.vs;
  const int mcux = (fr.W + 8 * hs - 1) / (8 * hs), mcuy = (fr.H + 8 * vs - 1) / (8 * vs);
  const int nluma = hs * vs, nb = nluma + 2;
  const int bw0 = mcux * hs;
  const int64_t base0 = fr.coef_off, base1 = base0 + static_cast<int64_t>(mcux) * hs * mcuy * vs;
  const int64_t base2 = base1 + static_cast<int64_t>(mcux) * mcuy;
  // table numbers of the three components, 4 bits each (no per-thread arrays: they would live in local memory)
  const int dct = (tb->comp_dc[0] & 1) | (tb->comp_dc[1] & 1) << 4 | (tb->comp_dc[2] & 1) << 8;
  const int act = (2 + (tb->comp_ac[0] & 1)) | (2 + (tb->comp_ac[1] & 1)) << 4 | (2 + (tb->comp_ac[2] & 1)) << 8;

  const uint8_t* seg = data + fr.seg_off;
  const int64_t seg_len = fr.seg_len;
  int64_t in_pos = 0;       // input bytes staged (all lanes)
  int64_t staged = 0;       // unstuffed bytes in the ring so far (all lanes)
  BitReader br{0ull, 0, 0, sm.ring};
  int pred0 = 0, pred1 = 0, pred2 = 0;       // DC predictors
  int err = X3D_JPEG_OK;
  __syncwarp();

  const int nmcu = mcux * mcuy;
  for (int m = 0; m < nmcu; ++m) {
    // ---- refill (warp-uniform decision on lane 0's read position)
    const int64_t rpos = __shfl_sync(0xffffffffu, br.rpos, 0);
    while (in_pos < seg_len && staged - rpos < kAhead) {
      uint8_t prev = in_pos > 0 ? __ldg(seg + in_pos - 1) : 0;
      for (int k = 0; k < kChunk / 32; ++k) {
        const int64_t i = in_pos + k * 32 + lane;
        const bool in = i < seg_len;
        const uint8_t b = in ? __ldg(seg + i) : 0;
        uint8_t before = __shfl_up_sync(0xffffffffu, b, 1);
        if (lane == 0) before = prev;
        prev = __shfl_sync(0xffffffffu, b, 31);
        const bool keep = in && !(b == 0 && before == 0xff);
        const uint32_t mask = __ballot_sync(0xffffffffu, keep);
        if (keep) sm.ring[(staged + __popc(mask & ((1u << lane) - 1u))) & (kRing - 1)] = b;
        staged += __popc(mask);
      }
      in_pos += kChunk;
      __syncwarp();
    }
    const int64_t avail = in_pos >= seg_len ? staged : INT64_MAX;   // zeros only past the real end

    // ---- lane 0 decodes one MCU
    if (lane == 0) {
      for (int b = 0; b < nb && err == X3D_JPEG_OK; ++b) {
        const int c = b < nluma ? 0 : b - nluma + 1;
        int16_t* blk = sm.blk[b];
        int s = huff_decode(br, avail, sm.h, (dct >> (4 * c)) & 15);
        if (s < 0) { err = X3D_JPEG_BAD_CODE; break; }
        if (s) s = huff_extend(get_bits(br, avail, s), s);
        const int pred = static_cast<int>(static_cast<uint32_t>(c == 0 ? pred0 : (c == 1 ? pred1 : pred2)) +
                                          static_cast<uint32_t>(s));
        if (c == 0) pred0 = pred; else if (c == 1) pred1 = pred; else pred2 = pred;
        blk[0] = static_cast<int16_t>(pred);
        const int t = (act >> (4 * c)) & 15;
        for (int k = 1; k < 64; ++k) {
          s = huff_decode(br, avail, sm.h, t);
          if (s < 0) { err = X3D_JPEG_BAD_CODE; break; }
          const int r = s >> 4;
          s &= 15;
          if (s) {
            k += r;
            if (k > 63) { err = X3D_JPEG_BAD_RUN; break; }
            blk[kNatural[k]] = static_cast<int16_t>(huff_extend(get_bits(br, avail, s), s));
          } else {
            if (r != 15) break;                                     // EOB
            k += 15;
            if (k > 63) { err = X3D_JPEG_BAD_RUN; break; }
          }
        }
      }
      // bits taken from the zeros past the segment's end
      if (err == X3D_JPEG_OK && in_pos >= seg_len && (br.rpos - staged) * 8 > br.nbits) err = X3D_JPEG_SHORT_DATA;
    }
    err = __shfl_sync(0xffffffffu, err, 0);
    __syncwarp();
    if (err != X3D_JPEG_OK) break;

    // ---- flush: nb blocks of 128 bytes, 16 bytes per lane and step, then zero them again
    const int my = m / mcux, mx = m - my * mcux;
    for (int i = lane; i < nb * 8; i += 32) {
      const int b = i >> 3, q = i & 7;
      int64_t blkno;
      if (b < nluma) blkno = base0 + static_cast<int64_t>(my * vs + b / hs) * bw0 + mx * hs + b % hs;
      else blkno = (b == nluma ? base1 : base2) + static_cast<int64_t>(my) * mcux + mx;
      int4* src = reinterpret_cast<int4*>(sm.blk[b]) + q;
      reinterpret_cast<int4*>(coef + blkno * 64)[q] = *src;
      *src = make_int4(0, 0, 0, 0);
    }
    __syncwarp();
  }
  if (lane == 0) status[fr.status] = err;
}

// ---------------------------------------------------------------------------------------------
// Stage 1 for restart intervals: one thread per interval, reading its bytes straight from global
// memory (each thread walks its own range sequentially, so the lines it touches stay in L1) and
// dropping the 00 stuffed after every FF.  A block is decoded into the thread's zeroed slot in shared
// memory and stored as eight 16-byte words.  The Huffman tables are read through the read-only cache:
// the intervals of one CTA may belong to frames with different tables.
constexpr int kRstThreads = 64;

struct RstReader {
  uint64_t acc;        // MSB-aligned
  int nbits;
  int32_t pos;         // next byte of the interval
  int32_t zeros;       // zero bytes appended past the interval's end
  const uint8_t* p;
  int32_t len;

  __device__ __forceinline__ void fill() {
    while (nbits <= 56) {
      uint32_t b = 0;
      if (pos < len) {
        b = __ldg(p + pos);
        pos += (b == 0xFF) ? 2 : 1;                 // FF 00 -> FF (a range never ends inside FF 00)
      } else {
        ++zeros;
      }
      acc |= static_cast<uint64_t>(b) << (56 - nbits);
      nbits += 8;
    }
  }
  __device__ __forceinline__ uint32_t peek(int n) const { return static_cast<uint32_t>(acc >> (64 - n)); }
  __device__ __forceinline__ void skip(int n) { acc <<= n; nbits -= n; }
  // bits were taken from the zeros past the end
  __device__ __forceinline__ bool overran() const { return zeros * 8 > nbits; }
};

__device__ __forceinline__ int rst_huff_decode(RstReader& br, const x3d_jpeg_huff* __restrict__ h) {
  br.fill();
  const uint32_t look = __ldg(&h->lookup[br.peek(8)]);
  int l = look >> 8;
  if (l <= 8) {
    br.skip(l);
    return look & 0xff;
  }
  int32_t code = static_cast<int32_t>(br.peek(9));
  l = 9;
  while (l <= 16 && code > __ldg(&h->maxcode[l])) {
    ++l;
    code = static_cast<int32_t>(br.peek(l));
  }
  if (l > 16) return -1;
  br.skip(l);
  return __ldg(&h->huffval[(code + __ldg(&h->valoffset[l])) & 0xff]);
}

__device__ __forceinline__ int rst_get_bits(RstReader& br, int s) {
  br.fill();
  const int r = static_cast<int>(br.peek(s));
  br.skip(s);
  return r;
}

__global__ void __launch_bounds__(kRstThreads)
entropy_rst_kernel(const uint8_t* __restrict__ data, const x3d_jpeg_frame* __restrict__ frames,
                   const x3d_jpeg_tables* __restrict__ tables, const x3d_jpeg_interval* __restrict__ intervals,
                   int nintervals, int16_t* __restrict__ coef, int32_t* __restrict__ status) {
  __shared__ __align__(16) int16_t blk_s[kRstThreads][64];
  const int i = blockIdx.x * kRstThreads + threadIdx.x;
  int4* slot = reinterpret_cast<int4*>(blk_s[threadIdx.x]);
#pragma unroll
  for (int q = 0; q < 8; ++q) slot[q] = make_int4(0, 0, 0, 0);
  if (i >= nintervals) return;
  const x3d_jpeg_interval iv = intervals[i];
  const x3d_jpeg_frame fr = frames[iv.frame];
  const x3d_jpeg_tables* tb = tables + fr.tables;
  const int hs = fr.hs, vs = fr.vs;
  const int mcux = (fr.W + 8 * hs - 1) / (8 * hs), mcuy = (fr.H + 8 * vs - 1) / (8 * vs);
  const int nluma = hs * vs, nb = nluma + 2;
  const int bw0 = mcux * hs;
  const int64_t base0 = fr.coef_off, base1 = base0 + static_cast<int64_t>(mcux) * hs * mcuy * vs;
  const int64_t base2 = base1 + static_cast<int64_t>(mcux) * mcuy;
  // table ids of the three components, one bit each (no per-thread arrays: they would live in local memory)
  const int dct = (tb->comp_dc[0] & 1) | (tb->comp_dc[1] & 1) << 1 | (tb->comp_dc[2] & 1) << 2;
  const int act = (tb->comp_ac[0] & 1) | (tb->comp_ac[1] & 1) << 1 | (tb->comp_ac[2] & 1) << 2;
  int16_t* blk = blk_s[threadIdx.x];
  RstReader br{0ull, 0, 0, 0, data + iv.off, iv.len};
  int pred0 = 0, pred1 = 0, pred2 = 0;       // DC predictors restart at 0 in every interval
  int err = X3D_JPEG_OK;
  for (int m = iv.mcu0; m < iv.mcu0 + iv.nmcu && err == X3D_JPEG_OK; ++m) {
    const int my = m / mcux, mx = m - my * mcux;
    for (int b = 0; b < nb; ++b) {
      const int c = b < nluma ? 0 : b - nluma + 1;
      int s = rst_huff_decode(br, &tb->dc[(dct >> c) & 1]);
      if (s < 0) { err = X3D_JPEG_BAD_CODE; break; }
      if (s) s = huff_extend(rst_get_bits(br, s), s);
      const int pred = static_cast<int>(static_cast<uint32_t>(c == 0 ? pred0 : (c == 1 ? pred1 : pred2)) +
                                        static_cast<uint32_t>(s));
      if (c == 0) pred0 = pred; else if (c == 1) pred1 = pred; else pred2 = pred;
      blk[0] = static_cast<int16_t>(pred);
      const x3d_jpeg_huff* at = &tb->ac[(act >> c) & 1];
      for (int k = 1; k < 64; ++k) {
        s = rst_huff_decode(br, at);
        if (s < 0) { err = X3D_JPEG_BAD_CODE; break; }
        const int r = s >> 4;
        s &= 15;
        if (s) {
          k += r;
          if (k > 63) { err = X3D_JPEG_BAD_RUN; break; }
          blk[kNatural[k]] = static_cast<int16_t>(huff_extend(rst_get_bits(br, s), s));
        } else {
          if (r != 15) break;                                       // EOB
          k += 15;
          if (k > 63) { err = X3D_JPEG_BAD_RUN; break; }
        }
      }
      if (err == X3D_JPEG_OK && br.overran()) err = X3D_JPEG_SHORT_DATA;
      if (err != X3D_JPEG_OK) break;
      int64_t blkno;
      if (b < nluma) blkno = base0 + static_cast<int64_t>(my * vs + b / hs) * bw0 + mx * hs + b % hs;
      else blkno = (b == nluma ? base1 : base2) + static_cast<int64_t>(my) * mcux + mx;
      int4* dst = reinterpret_cast<int4*>(coef + blkno * 64);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        dst[q] = slot[q];
        slot[q] = make_int4(0, 0, 0, 0);
      }
    }
  }
  if (err != X3D_JPEG_OK) atomicMax(status + fr.status, err);
}

// ---------------------------------------------------------------------------------------------
// Stage 2: IDCT.  A CTA takes 32 consecutive blocks of one frame; thread (block, r) runs column r of
// pass 1 and row r of pass 2 and stores the row's 8 samples with one 8-byte store.  The arithmetic
// is libjpeg's with JLONG = 64-bit, so even pathological coefficients give libjpeg's result.
constexpr int kIdctBlocks = 32;

__device__ __forceinline__ int64_t descale(int64_t x, int n) { return (x + (int64_t(1) << (n - 1))) >> n; }

// IDCT_range_limit(cinfo)[x & RANGE_MASK]: x + 128 clamped to [0, 255], x taken modulo 1024 in [-512, 511]
__device__ __forceinline__ uint32_t idct_limit(int64_t x) {
  const int v = static_cast<int>((x + 512) & 1023) - 512 + 128;
  return static_cast<uint32_t>(min(max(v, 0), 255));
}

// jidctint.c jpeg_idct_islow, one column (pass 1) or row (pass 2) of 8 values
template <bool kPass2>
__device__ __forceinline__ void islow_1d(const int64_t (&in)[8], int64_t (&out)[8]) {
  constexpr int CB = 13, P1 = 2;
  int64_t z2 = in[2], z3 = in[6];
  int64_t z1 = (z2 + z3) * 4433;
  const int64_t tmp2a = z1 + z3 * -15137, tmp3a = z1 + z2 * 6270;
  z2 = in[0]; z3 = in[4];
  const int64_t tmp0a = (z2 + z3) * (int64_t(1) << CB), tmp1a = (z2 - z3) * (int64_t(1) << CB);
  const int64_t tmp10 = tmp0a + tmp3a, tmp13 = tmp0a - tmp3a, tmp11 = tmp1a + tmp2a, tmp12 = tmp1a - tmp2a;
  int64_t tmp0 = in[7], tmp1 = in[5], tmp2 = in[3], tmp3 = in[1];
  z1 = tmp0 + tmp3; z2 = tmp1 + tmp2; z3 = tmp0 + tmp2;
  int64_t z4 = tmp1 + tmp3;
  const int64_t z5 = (z3 + z4) * 9633;
  tmp0 *= 2446; tmp1 *= 16819; tmp2 *= 25172; tmp3 *= 12299;
  z1 *= -7373; z2 *= -20995; z3 *= -16069; z4 *= -3196;
  z3 += z5; z4 += z5;
  tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
  constexpr int n = kPass2 ? CB + P1 + 3 : CB - P1;
  out[0] = descale(tmp10 + tmp3, n); out[7] = descale(tmp10 - tmp3, n);
  out[1] = descale(tmp11 + tmp2, n); out[6] = descale(tmp11 - tmp2, n);
  out[2] = descale(tmp12 + tmp1, n); out[5] = descale(tmp12 - tmp1, n);
  out[3] = descale(tmp13 + tmp0, n); out[4] = descale(tmp13 - tmp0, n);
}

// jidctfst.c jpeg_idct_ifast (DCTELEM = int, MULTIPLY descaled by 8 without rounding)
__device__ __forceinline__ int32_t fmul(int32_t v, int32_t c) { return static_cast<int32_t>((static_cast<int64_t>(v) * c) >> 8); }

__device__ __forceinline__ void ifast_1d(const int32_t (&in)[8], int32_t (&out)[8]) {
  int32_t tmp0 = in[0], tmp1 = in[2], tmp2 = in[4], tmp3 = in[6];
  int32_t tmp10 = tmp0 + tmp2, tmp11 = tmp0 - tmp2, tmp13 = tmp1 + tmp3;
  int32_t tmp12 = fmul(tmp1 - tmp3, 362) - tmp13;
  tmp0 = tmp10 + tmp13; tmp3 = tmp10 - tmp13; tmp1 = tmp11 + tmp12; tmp2 = tmp11 - tmp12;
  const int32_t tmp4i = in[1], tmp5i = in[3], tmp6i = in[5], tmp7i = in[7];
  const int32_t z13 = tmp6i + tmp5i, z10 = tmp6i - tmp5i, z11 = tmp4i + tmp7i, z12 = tmp4i - tmp7i;
  const int32_t tmp7 = z11 + z13;
  tmp11 = fmul(z11 - z13, 362);
  const int32_t z5 = fmul(z10 + z12, 473);
  tmp10 = fmul(z12, 277) - z5;
  tmp12 = fmul(z10, -669) + z5;
  const int32_t tmp6 = tmp12 - tmp7, tmp5 = tmp11 - tmp6, tmp4 = tmp10 + tmp5;
  out[0] = tmp0 + tmp7; out[7] = tmp0 - tmp7; out[1] = tmp1 + tmp6; out[6] = tmp1 - tmp6;
  out[2] = tmp2 + tmp5; out[5] = tmp2 - tmp5; out[4] = tmp3 + tmp4; out[3] = tmp3 - tmp4;
}

template <int kMethod>
__global__ void __launch_bounds__(kIdctBlocks * 8)
idct_kernel(const int16_t* __restrict__ coef, const x3d_jpeg_frame* __restrict__ frames,
            const x3d_jpeg_tables* __restrict__ tables, uint8_t* __restrict__ planes) {
  __shared__ __align__(16) int16_t cs[kIdctBlocks][64];
  __shared__ int32_t ws[kIdctBlocks][64];
  const x3d_jpeg_frame fr = frames[blockIdx.y];
  const int mcux = (fr.W + 8 * fr.hs - 1) / (8 * fr.hs), mcuy = (fr.H + 8 * fr.vs - 1) / (8 * fr.vs);
  const int bw0 = mcux * fr.hs, n0 = bw0 * mcuy * fr.vs, n1 = mcux * mcuy;
  const int nblocks = n0 + 2 * n1;
  const int first = blockIdx.x * kIdctBlocks;
  if (first >= nblocks) return;
  const int tid = threadIdx.x;
  {
    const int b = first + (tid >> 3);                     // 256 threads x 16 bytes = 32 blocks
    if (b < nblocks)
      reinterpret_cast<int4*>(&cs[0][0])[tid] = reinterpret_cast<const int4*>(coef + (fr.coef_off + first) * 64)[tid];
  }
  __syncthreads();
  const int lb = tid >> 3, r = tid & 7, b = first + lb;
  const bool live = b < nblocks;
  const int c = b < n0 ? 0 : (b < n0 + n1 ? 1 : 2);
  const uint16_t* q = tables[fr.tables].q[tables[fr.tables].comp_q[c]];
  if (kMethod == X3D_JPEG_ISLOW) {
    int64_t in[8], out[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) in[i] = live ? int64_t(cs[lb][i * 8 + r]) * int64_t(q[i * 8 + r]) : 0;
    islow_1d<false>(in, out);
#pragma unroll
    for (int i = 0; i < 8; ++i) ws[lb][i * 8 + r] = static_cast<int32_t>(out[i]);
  } else {
    int32_t in[8], out[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int k = i * 8 + r;
      const int32_t mult = live ? static_cast<int32_t>((int32_t(q[k]) * kAanScales[k] + 2048) >> 12) : 0;
      in[i] = int32_t(cs[lb][k]) * mult;
    }
    ifast_1d(in, out);
#pragma unroll
    for (int i = 0; i < 8; ++i) ws[lb][i * 8 + r] = out[i];
  }
  __syncthreads();
  if (!live) return;
  uint32_t px[8];
  if (kMethod == X3D_JPEG_ISLOW) {
    int64_t in[8], out[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) in[i] = ws[lb][r * 8 + i];
    islow_1d<true>(in, out);
#pragma unroll
    for (int i = 0; i < 8; ++i) px[i] = idct_limit(out[i]);
  } else {
    int32_t in[8], out[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) in[i] = ws[lb][r * 8 + i];
    ifast_1d(in, out);
#pragma unroll
    for (int i = 0; i < 8; ++i) px[i] = idct_limit(out[i] >> 5);        // IDESCALE(x, PASS1_BITS + 3)
  }
  // block position in its component's plane
  int bw, bi;
  int64_t pbase = fr.plane_off;
  if (c == 0) { bw = bw0; bi = b; }
  else {
    bw = mcux;
    bi = b - n0 - (c - 1) * n1;
    pbase += static_cast<int64_t>(n0) * 64 + static_cast<int64_t>(c - 1) * n1 * 64;
  }
  const int by = bi / bw, bx = bi - by * bw;
  uint8_t* dst = planes + pbase + (static_cast<int64_t>(by) * 8 + r) * (bw * 8) + bx * 8;
  *reinterpret_cast<uint2*>(dst) = make_uint2(px[0] | px[1] << 8 | px[2] << 16 | px[3] << 24,
                                              px[4] | px[5] << 8 | px[6] << 16 | px[7] << 24);
}

// ---------------------------------------------------------------------------------------------
// Stage 3: chroma upsampling and YCbCr -> RGB, four output pixels (12 bytes) per thread.
// jdcolor.c build_ycc_rgb_table with SCALEBITS 16:
//   R = y + ((91881 * (cr-128) + 32768) >> 16);  B = y + ((116130 * (cb-128) + 32768) >> 16)
//   G = y + ((-22554 * (cb-128) + 32768 - 46802 * (cr-128)) >> 16);   each clamped to [0, 255]
constexpr int kColorThreads = 256;

struct Planes {
  const uint8_t* p;
  int w, dw, dh;        // plane row pitch, downsampled extent
};

// chroma sample at output pixel (y, x) of a 2x1 frame: jdsample.c h2v1_fancy_upsample (fancy = 1) or
// h2v1_upsample (fancy = 0, two columns or fewer)
__device__ __forceinline__ int chroma_h2v1(const Planes& pl, int y, int x, bool fancy) {
  const uint8_t* r = pl.p + static_cast<int64_t>(y) * pl.w;
  const int j = x >> 1;
  if (!fancy) return r[j];
  if (x & 1) return j == pl.dw - 1 ? r[j] : (r[j] * 3 + r[j + 1] + 2) >> 2;
  return j == 0 ? r[0] : (r[j] * 3 + r[j - 1] + 1) >> 2;
}

// chroma sample at output pixel (y, x): jdsample.c h2v2_fancy_upsample (fancy = 1), h2v2_upsample
// (fancy = 0, two columns or fewer), or the sample itself (1x1 luma)
__device__ __forceinline__ int chroma(const Planes& pl, int y, int x, int up, bool fancy) {
  if (!up) return pl.p[static_cast<int64_t>(y) * pl.w + x];
  const int i = y >> 1, j = x >> 1;
  if (!fancy) return pl.p[static_cast<int64_t>(i) * pl.w + j];
  const int far_row = (y & 1) ? min(i + 1, pl.dh - 1) : max(i - 1, 0);
  const uint8_t* r0 = pl.p + static_cast<int64_t>(i) * pl.w;
  const uint8_t* r1 = pl.p + static_cast<int64_t>(far_row) * pl.w;
  const int jn = (x & 1) ? min(j + 1, pl.dw - 1) : max(j - 1, 0);
  const int cs = r0[j] * 3 + r1[j], cn = r0[jn] * 3 + r1[jn];
  return (x & 1) ? (cs * 3 + cn + 7) >> 4 : (cs * 3 + cn + 8) >> 4;
}

__device__ __forceinline__ uint32_t clamp255(int v) { return static_cast<uint32_t>(min(max(v, 0), 255)); }

__global__ void __launch_bounds__(kColorThreads)
color_kernel(const uint8_t* __restrict__ planes, const x3d_jpeg_frame* __restrict__ frames,
             uint8_t* __restrict__ out) {
  const x3d_jpeg_frame fr = frames[blockIdx.y];
  const int64_t npix = static_cast<int64_t>(fr.H) * fr.W;
  const int64_t p0 = (static_cast<int64_t>(blockIdx.x) * kColorThreads + threadIdx.x) * 4;
  if (p0 >= npix) return;
  const int hs = fr.hs, vs = fr.vs;
  const int mcux = (fr.W + 8 * hs - 1) / (8 * hs), mcuy = (fr.H + 8 * vs - 1) / (8 * vs);
  const int w0 = mcux * hs * 8, w1 = mcux * 8;
  const int up = hs == 2;
  const bool h2v1 = up && vs == 1;                 // 4:2:2 (Motion-JPEG frames)
  Planes cb, cr;
  cb.p = planes + fr.plane_off + static_cast<int64_t>(w0) * mcuy * vs * 8;
  cr.p = cb.p + static_cast<int64_t>(w1) * mcuy * 8;
  cb.w = cr.w = w1;
  cb.dw = cr.dw = up ? (fr.W + 1) >> 1 : fr.W;
  cb.dh = cr.dh = up && !h2v1 ? (fr.H + 1) >> 1 : fr.H;
  const bool fancy = cb.dw > 2;
  const uint8_t* yp = planes + fr.plane_off;
  uint32_t v[12];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int64_t p = min(p0 + k, npix - 1);
    const int y = static_cast<int>(p / fr.W), x = static_cast<int>(p - static_cast<int64_t>(y) * fr.W);
    const int Y = yp[static_cast<int64_t>(y) * w0 + x];
    const int Cb = (h2v1 ? chroma_h2v1(cb, y, x, fancy) : chroma(cb, y, x, up, fancy)) - 128;
    const int Cr = (h2v1 ? chroma_h2v1(cr, y, x, fancy) : chroma(cr, y, x, up, fancy)) - 128;
    v[3 * k + 0] = clamp255(Y + ((91881 * Cr + 32768) >> 16));
    v[3 * k + 1] = clamp255(Y + ((-22554 * Cb + 32768 - 46802 * Cr) >> 16));
    v[3 * k + 2] = clamp255(Y + ((116130 * Cb + 32768) >> 16));
  }
  uint8_t* o = out + fr.out_off + p0 * 3;
  if (p0 + 4 <= npix) {
    uint32_t* o32 = reinterpret_cast<uint32_t*>(o);
#pragma unroll
    for (int w = 0; w < 3; ++w) o32[w] = v[4 * w] | (v[4 * w + 1] << 8) | (v[4 * w + 2] << 16) | (v[4 * w + 3] << 24);
  } else {
    const int nb = static_cast<int>(npix - p0) * 3;
#pragma unroll
    for (int b = 0; b < 12; ++b)
      if (b < nb) o[b] = static_cast<uint8_t>(v[b]);
  }
}

}  // namespace jpeg
}  // namespace x3d

using namespace x3d;

extern "C" int x3d_jpeg_entropy(const uint8_t* data, const x3d_jpeg_frame* frames, const x3d_jpeg_tables* tables,
                                int nframes, int16_t* coef, int32_t* status, void* stream) {
  X3D_REQUIRE(data && frames && tables && coef && status, X3D_ERR_INVALID_ARG, "x3d_jpeg_entropy: null pointer");
  X3D_REQUIRE(nframes > 0, X3D_ERR_INVALID_ARG, "x3d_jpeg_entropy: nframes=%d", nframes);
  X3D_REQUIRE((reinterpret_cast<uintptr_t>(coef) & 15) == 0 && (reinterpret_cast<uintptr_t>(frames) & 7) == 0 &&
              (reinterpret_cast<uintptr_t>(tables) & 3) == 0 && (reinterpret_cast<uintptr_t>(status) & 3) == 0,
              X3D_ERR_INVALID_ARG, "x3d_jpeg_entropy: coef must be 16-byte, frames 8-byte, tables/status 4-byte aligned");
  jpeg::entropy_kernel<<<nframes, 32, 0, static_cast<cudaStream_t>(stream)>>>(data, frames, tables, coef, status);
  return check_launch("x3d_jpeg_entropy");
}

extern "C" int x3d_jpeg_entropy_rst(const uint8_t* data, const x3d_jpeg_frame* frames, const x3d_jpeg_tables* tables,
                                    const x3d_jpeg_interval* intervals, int nintervals, int16_t* coef, int32_t* status,
                                    void* stream) {
  X3D_REQUIRE(data && frames && tables && intervals && coef && status, X3D_ERR_INVALID_ARG,
              "x3d_jpeg_entropy_rst: null pointer");
  X3D_REQUIRE(nintervals > 0, X3D_ERR_INVALID_ARG, "x3d_jpeg_entropy_rst: nintervals=%d", nintervals);
  X3D_REQUIRE((reinterpret_cast<uintptr_t>(coef) & 15) == 0 && (reinterpret_cast<uintptr_t>(frames) & 7) == 0 &&
              (reinterpret_cast<uintptr_t>(intervals) & 7) == 0 && (reinterpret_cast<uintptr_t>(tables) & 3) == 0 &&
              (reinterpret_cast<uintptr_t>(status) & 3) == 0,
              X3D_ERR_INVALID_ARG,
              "x3d_jpeg_entropy_rst: coef must be 16-byte, frames/intervals 8-byte, tables/status 4-byte aligned");
  const int grid = (nintervals + jpeg::kRstThreads - 1) / jpeg::kRstThreads;
  jpeg::entropy_rst_kernel<<<grid, jpeg::kRstThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      data, frames, tables, intervals, nintervals, coef, status);
  return check_launch("x3d_jpeg_entropy_rst");
}

extern "C" int x3d_jpeg_idct(const int16_t* coef, const x3d_jpeg_frame* frames, const x3d_jpeg_tables* tables,
                             int nframes, int max_blocks, int method, uint8_t* planes, void* stream) {
  X3D_REQUIRE(coef && frames && tables && planes, X3D_ERR_INVALID_ARG, "x3d_jpeg_idct: null pointer");
  X3D_REQUIRE(nframes > 0 && nframes <= 65535 && max_blocks > 0, X3D_ERR_INVALID_ARG,
              "x3d_jpeg_idct: nframes=%d (1..65535) max_blocks=%d", nframes, max_blocks);
  X3D_REQUIRE(method == X3D_JPEG_ISLOW || method == X3D_JPEG_IFAST, X3D_ERR_INVALID_ARG, "x3d_jpeg_idct: method %d", method);
  X3D_REQUIRE((reinterpret_cast<uintptr_t>(coef) & 15) == 0 && (reinterpret_cast<uintptr_t>(planes) & 7) == 0 &&
              (reinterpret_cast<uintptr_t>(frames) & 7) == 0 && (reinterpret_cast<uintptr_t>(tables) & 3) == 0,
              X3D_ERR_INVALID_ARG, "x3d_jpeg_idct: coef must be 16-byte, planes/frames 8-byte, tables 4-byte aligned");
  const dim3 grid((max_blocks + jpeg::kIdctBlocks - 1) / jpeg::kIdctBlocks, nframes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (method == X3D_JPEG_ISLOW)
    jpeg::idct_kernel<X3D_JPEG_ISLOW><<<grid, jpeg::kIdctBlocks * 8, 0, st>>>(coef, frames, tables, planes);
  else
    jpeg::idct_kernel<X3D_JPEG_IFAST><<<grid, jpeg::kIdctBlocks * 8, 0, st>>>(coef, frames, tables, planes);
  return check_launch("x3d_jpeg_idct");
}

extern "C" int x3d_jpeg_color(const uint8_t* planes, const x3d_jpeg_frame* frames, int nframes, int64_t max_pixels,
                              uint8_t* out, void* stream) {
  X3D_REQUIRE(planes && frames && out, X3D_ERR_INVALID_ARG, "x3d_jpeg_color: null pointer");
  X3D_REQUIRE(nframes > 0 && nframes <= 65535 && max_pixels > 0, X3D_ERR_INVALID_ARG,
              "x3d_jpeg_color: nframes=%d (1..65535) max_pixels=%lld", nframes, (long long)max_pixels);
  X3D_REQUIRE((reinterpret_cast<uintptr_t>(out) & 3) == 0 && (reinterpret_cast<uintptr_t>(frames) & 7) == 0,
              X3D_ERR_INVALID_ARG, "x3d_jpeg_color: out must be 4-byte, frames 8-byte aligned");
  const int64_t gx = ((max_pixels + 3) / 4 + jpeg::kColorThreads - 1) / jpeg::kColorThreads;
  X3D_REQUIRE(gx <= 0x7fffffffLL, X3D_ERR_UNSUPPORTED, "x3d_jpeg_color: max_pixels=%lld", (long long)max_pixels);
  const dim3 grid(static_cast<unsigned>(gx), nframes);
  jpeg::color_kernel<<<grid, jpeg::kColorThreads, 0, static_cast<cudaStream_t>(stream)>>>(planes, frames, out);
  return check_launch("x3d_jpeg_color");
}
