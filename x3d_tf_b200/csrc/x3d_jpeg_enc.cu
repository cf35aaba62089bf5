// Baseline JPEG encoding of video frames (the reference's tf.io.encode_jpeg in
// datasets/create_tfrecords.py:48-83), reproducing libjpeg-turbo's compressor with TF's settings
// (JDCT_ISLOW, standard Huffman tables, no restart interval) bit for bit, in four calls per ragged
// batch of frames:
//   x3d_jpeg_fdct      jccolor.c + jcsample.c + jfdctint.c + jcdctmgr.c     -> int16 coefficient blocks
//   x3d_jpeg_enc_bits  jchuff.c code lengths of every block, exclusive scan  -> bit offset of every block
//   x3d_jpeg_enc_emit  jchuff.c encode_one_block at those offsets            -> 32-bit words of bits
//   x3d_jpeg_enc_stuff flush_bits' byte stuffing (FF -> FF 00)               -> entropy-coded segments
//                      (two kernels: the segments' offsets, then the stuffing)
// Unlike decoding, every block's code is independent of the others once the DC predictions are known
// (the previous block's quantised DC), so no stage has a serial chain.  Layouts: include/x3d_b200.h.
#include <cub/block/block_scan.cuh>

#include "common.cuh"

namespace x3d {
namespace jpeg_enc {

// zigzag position -> natural index (ITU T.81 figure A.6)
__constant__ uint8_t kZigzag[64] = {
    0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
    41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
    30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

struct Grid {
  int hs, mcux, mcuy, bw0, n0, n1, nblocks, nb;      // nb blocks per MCU
  __device__ explicit Grid(const x3d_jpeg_enc_frame& fr) {
    hs = fr.hs;
    mcux = (fr.W + 8 * hs - 1) / (8 * hs);
    mcuy = (fr.H + 8 * hs - 1) / (8 * hs);
    bw0 = mcux * hs;
    n0 = bw0 * mcuy * hs;
    n1 = mcux * mcuy;
    nblocks = n0 + 2 * n1;
    nb = hs * hs + 2;
  }
  // storage index (the decoder's layout) and component of the block at scan position s
  __device__ __forceinline__ int block(int s, int& c) const {
    const int m = s / nb, k = s - m * nb, my = m / mcux, mx = m - my * mcux;
    const int nl = nb - 2;
    if (k < nl) { c = 0; return (my * hs + k / hs) * bw0 + mx * hs + k % hs; }
    c = k - nl + 1;
    return n0 + (c - 1) * n1 + m;
  }
  // storage index of the same component's block before scan position s, or -1 for the first
  __device__ __forceinline__ int prev_block(int s) const {
    const int k = s % nb, nl = nb - 2;
    int c;
    if (k > 0 && k < nl) return block(s - 1, c);          // previous luma block of this MCU
    if (s < nb) return -1;                                 // first MCU
    return block(s - nb + (k == 0 ? nl - 1 : 0), c);       // last luma block / same chroma of MCU m-1
  }
};

// ---------------------------------------------------------------------------------------------
// Stage A: colour conversion, downsampling, forward DCT and quantisation.  A CTA takes 32 blocks of
// one frame; thread (block, r) converts and transforms row r (pass 1), then column r (pass 2).
constexpr int kFdctBlocks = 32;

// jccolor.c rgb_ycc_start: SCALEBITS 16, FIX(x) = x * 65536 + 0.5; Y rounds with ONE_HALF, Cb / Cr
// add CBCR_OFFSET + ONE_HALF - 1 (so that 255 cannot round up to 256)
__device__ __forceinline__ int ycc(const uint8_t* p, int c) {
  const int r = p[0], g = p[1], b = p[2];
  if (c == 0) return (19595 * r + 38470 * g + 7471 * b + 32768) >> 16;
  if (c == 1) return (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16;
  return (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16;
}

// jfdctint.c jpeg_fdct_islow, one row (pass 1) or column (pass 2); DESCALE rounds half up
__device__ __forceinline__ int descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }

template <bool kPass2>
__device__ __forceinline__ void fdct_1d(const int (&d)[8], int (&o)[8]) {
  constexpr int CB = 13, P1 = 2, n = kPass2 ? CB + P1 : CB - P1;
  const int tmp0 = d[0] + d[7], tmp7 = d[0] - d[7], tmp1 = d[1] + d[6], tmp6 = d[1] - d[6];
  const int tmp2 = d[2] + d[5], tmp5 = d[2] - d[5], tmp3 = d[3] + d[4], tmp4 = d[3] - d[4];
  const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
  if (kPass2) { o[0] = descale(tmp10 + tmp11, P1); o[4] = descale(tmp10 - tmp11, P1); }
  else { o[0] = (tmp10 + tmp11) * (1 << P1); o[4] = (tmp10 - tmp11) * (1 << P1); }
  int z1 = (tmp12 + tmp13) * 4433;
  o[2] = descale(z1 + tmp13 * 6270, n);
  o[6] = descale(z1 + tmp12 * -15137, n);
  z1 = tmp4 + tmp7;
  int z2 = tmp5 + tmp6, z3 = tmp4 + tmp6, z4 = tmp5 + tmp7;
  const int z5 = (z3 + z4) * 9633;
  z1 *= -7373; z2 *= -20995; z3 = z3 * -16069 + z5; z4 = z4 * -3196 + z5;
  o[7] = descale(tmp4 * 2446 + z1 + z3, n);
  o[5] = descale(tmp5 * 16819 + z2 + z4, n);
  o[3] = descale(tmp6 * 25172 + z2 + z3, n);
  o[1] = descale(tmp7 * 12299 + z1 + z4, n);
}

__global__ void __launch_bounds__(kFdctBlocks * 8)
fdct_kernel(const uint8_t* __restrict__ rgb, const x3d_jpeg_enc_frame* __restrict__ frames,
            const x3d_jpeg_enc_tables* __restrict__ tables, int16_t* __restrict__ coef) {
  __shared__ int32_t ws[kFdctBlocks][65];
  __shared__ __align__(16) int16_t cs[kFdctBlocks][64];
  __shared__ uint32_t recip[2][64];
  __shared__ uint32_t corr[2][64];
  __shared__ int32_t shift[2][64];
  const x3d_jpeg_enc_frame fr = frames[blockIdx.y];
  const Grid g(fr);
  const int first = blockIdx.x * kFdctBlocks;
  if (first >= g.nblocks) return;
  const int tid = threadIdx.x;
  if (tid < 128) {
    // jcdctmgr.c compute_reciprocal(quantval << 3) with the 16-bit DCTELEM of libjpeg-turbo's SIMD
    // build (what TF and Pillow link): quantize = sign(x) * (((|x| + corr) * recip) >> (shift + 16))
    const uint32_t d = static_cast<uint32_t>(tables[fr.tables].q[tid >> 6][tid & 63]) << 3;
    const int b = 31 - __clz(d);
    int r = 16 + b;
    uint32_t fq = (1u << r) / d, c = d / 2;
    const uint32_t fr_ = (1u << r) % d;
    if (fr_ == 0) { fq >>= 1; --r; }
    else if (fr_ <= d / 2) ++c;
    else ++fq;
    recip[tid >> 6][tid & 63] = fq;
    corr[tid >> 6][tid & 63] = c;
    shift[tid >> 6][tid & 63] = r;
  }
  const int lb = tid >> 3, r = tid & 7, b = min(first + lb, g.nblocks - 1);
  const int c = b < g.n0 ? 0 : (b < g.n0 + g.n1 ? 1 : 2);
  const int bw = c == 0 ? g.bw0 : g.mcux;
  const int bi = c == 0 ? b : b - g.n0 - (c - 1) * g.n1;
  int by = bi / bw, bx = bi - by * bw;
  // jccoefct.c compress_data: the blocks of the right / bottom MCUs past ceil(W/8) x ceil(H/8) (4:2:0
  // luma only) are dummy blocks, AC zero and DC that of the block before them in the MCU, which is
  // always the real block (min(bx | 1, wib - 1), min(by, hib - 1)); transform that one instead
  const int wib = (fr.W + 7) >> 3, hib = (fr.H + 7) >> 3;
  const bool dummy = c == 0 && (bx >= wib || by >= hib);
  if (dummy) { bx = min(bx | 1, wib - 1); by = min(by, hib - 1); }
  const uint8_t* img = rgb + fr.in_off;
  const int64_t pitch = static_cast<int64_t>(fr.W) * 3;
  int d[8], o[8];
  if (c == 0 || g.hs == 1) {
    // full-size component, last row / column replicated (jcprepct.c expand_bottom_edge,
    // jcsample.c expand_right_edge + fullsize_downsample)
    const int y = min(by * 8 + r, fr.H - 1);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int x = min(bx * 8 + k, fr.W - 1);
      d[k] = ycc(img + y * pitch + x * 3, c) - 128;
    }
  } else {
    // jcsample.c h2v2_downsample: (4 samples + bias) >> 2, bias 1, 2 alternating by output column;
    // columns replicated to 2 * width_in_blocks * 8, rows to even, then the last downsampled row
    // replicated to the iMCU height
    const int dh = (fr.H + 1) >> 1;
    const int i = min(by * 8 + r, dh - 1);
    const uint8_t* r0 = img + (2 * i) * pitch;
    const uint8_t* r1 = img + min(2 * i + 1, fr.H - 1) * pitch;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int x0 = min(2 * (bx * 8 + k), fr.W - 1) * 3, x1 = min(2 * (bx * 8 + k) + 1, fr.W - 1) * 3;
      d[k] = ((ycc(r0 + x0, c) + ycc(r0 + x1, c) + ycc(r1 + x0, c) + ycc(r1 + x1, c) + 1 + (k & 1)) >> 2) - 128;
    }
  }
  fdct_1d<false>(d, o);
#pragma unroll
  for (int k = 0; k < 8; ++k) ws[lb][r * 8 + k] = o[k];
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 8; ++k) d[k] = ws[lb][k * 8 + r];
  fdct_1d<true>(d, o);
  const int t = c == 0 ? 0 : 1;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int n = k * 8 + r;
    const uint32_t a = static_cast<uint32_t>(abs(o[k]));
    const int v = static_cast<int>(((a + corr[t][n]) * recip[t][n]) >> shift[t][n]);
    cs[lb][n] = static_cast<int16_t>(dummy && n != 0 ? 0 : (o[k] < 0 ? -v : v));
  }
  __syncthreads();
  // 256 threads x 16 bytes = 32 blocks of 128 bytes
  if (first + (tid >> 3) < g.nblocks)
    reinterpret_cast<int4*>(coef + (fr.coef_off + first) * 64)[tid] = reinterpret_cast<const int4*>(&cs[0][0])[tid];
}

// ---------------------------------------------------------------------------------------------
// Stages B and C: jchuff.c encode_one_block.  The walk over a block is the same for its length and
// its bits; Sink decides what happens to each (code, length).
struct EncSmem {
  uint16_t code[4][256];        // dc0, ac0, dc1, ac1
  uint8_t size[4][256];
};

__device__ __forceinline__ void load_tables(EncSmem& sm, const x3d_jpeg_enc_tables& t) {
  for (int i = threadIdx.x; i < 4 * 256; i += blockDim.x) {
    sm.code[i >> 8][i & 255] = t.code[i >> 8][i & 255];
    sm.size[i >> 8][i & 255] = t.size[i >> 8][i & 255];
  }
}

__device__ __forceinline__ int nbits(int a) { return 32 - __clz(a); }   // JPEG_NBITS, a >= 0

// calls put(code, length) with length <= 27 (a Huffman code and its value bits together)
template <typename Put>
__device__ __forceinline__ void encode_block(const int16_t* __restrict__ blk, int last_dc, int c,
                                             const EncSmem& sm, Put&& put) {
  const int dt = c == 0 ? 0 : 2, at = dt + 1;
  int t = blk[0] - last_dc;
  int a = abs(t), n = a ? nbits(a) : 0;
  // negative values send t - 1 in n bits (jchuff.c: temp2 += temp3)
  put((static_cast<uint32_t>(sm.code[dt][n]) << n) | (static_cast<uint32_t>(t < 0 ? t - 1 : t) & ((1u << n) - 1u)),
      sm.size[dt][n] + n);
  int run = 0;
  for (int k = 1; k < 64; ++k) {
    const int v = blk[kZigzag[k]];
    if (v == 0) { ++run; continue; }
    while (run > 15) { put(sm.code[at][0xF0], sm.size[at][0xF0]); run -= 16; }
    a = abs(v);
    n = nbits(a);
    const int s = (run << 4) + n;
    put((static_cast<uint32_t>(sm.code[at][s]) << n) | (static_cast<uint32_t>(v < 0 ? v - 1 : v) & ((1u << n) - 1u)),
        sm.size[at][s] + n);
    run = 0;
  }
  if (run > 0) put(sm.code[at][0], sm.size[at][0]);
}

// Stage B: one CTA per frame walks its blocks in scan order, kEncThreads at a time, and writes the
// exclusive bit offset of each (by scan position), the frame's bit count and status, and zeroes the
// words stage C ORs the bits into.
constexpr int kEncThreads = 512;

__global__ void __launch_bounds__(kEncThreads)
bits_kernel(const int16_t* __restrict__ coef, const x3d_jpeg_enc_frame* __restrict__ frames,
            const x3d_jpeg_enc_tables* __restrict__ tables, int64_t* __restrict__ boff,
            x3d_jpeg_enc_result* __restrict__ res, uint32_t* __restrict__ words) {
  using Scan = cub::BlockScan<int64_t, kEncThreads>;
  __shared__ typename Scan::TempStorage scan_tmp;
  __shared__ EncSmem sm;
  __shared__ int64_t carry;
  const x3d_jpeg_enc_frame fr = frames[blockIdx.x];
  const Grid g(fr);
  load_tables(sm, tables[fr.tables]);
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int16_t* cf = coef + fr.coef_off * 64;
  for (int s0 = 0; s0 < g.nblocks; s0 += kEncThreads) {
    const int s = s0 + threadIdx.x;
    int64_t len = 0;
    if (s < g.nblocks) {
      int c;
      const int b = g.block(s, c), p = g.prev_block(s);
      encode_block(cf + static_cast<int64_t>(b) * 64, p < 0 ? 0 : cf[static_cast<int64_t>(p) * 64], c, sm,
                   [&](uint32_t, int l) { len += l; });
    }
    int64_t excl, total;
    Scan(scan_tmp).ExclusiveSum(len, excl, total);
    const int64_t base = carry;
    if (s < g.nblocks) boff[fr.coef_off + s] = base + excl;
    __syncthreads();
    if (threadIdx.x == 0) carry = base + total;
    __syncthreads();
  }
  const int64_t bits = carry;
  const int64_t nwords = (bits + 31) >> 5;
  const bool fits = nwords <= fr.word_cap;
  if (threadIdx.x == 0) {
    res[blockIdx.x].bits = bits;
    res[blockIdx.x].status = fits ? X3D_JPEG_OK : X3D_JPEG_OVERFLOW;
  }
  if (fits)
    for (int64_t i = threadIdx.x; i < nwords; i += kEncThreads) words[fr.word_off + i] = 0u;
}

// Stage C1: one thread per block ORs its bits into the frame's words (MSB first: bit 0 of the stream
// is bit 31 of word 0).  Words wholly inside a block are stored; the two it may share with its
// neighbours are ORed atomically.  The frame's last block also pads to a byte with 1-bits.
constexpr int kEmitThreads = 256;

struct WordWriter {
  uint32_t* w;           // the word holding bit 0 of the block
  uint64_t acc;          // pending bits, right-aligned
  int nacc;              // pending bit count (< 32 between calls)
  int64_t wi;            // word the pending bits start in, relative to w
  __device__ __forceinline__ void put(uint32_t code, int len) {
    acc = (acc << len) | code;
    nacc += len;
    if (nacc >= 32) {
      const uint32_t word = static_cast<uint32_t>(acc >> (nacc - 32));
      if (wi == 0) atomicOr(w, word); else w[wi] = word;
      ++wi;
      nacc -= 32;
      acc &= (uint64_t(1) << nacc) - 1u;
    }
  }
  __device__ __forceinline__ void finish() {
    if (nacc > 0) atomicOr(w + wi, static_cast<uint32_t>(acc << (32 - nacc)));
  }
};

__global__ void __launch_bounds__(kEmitThreads)
emit_kernel(const int16_t* __restrict__ coef, const x3d_jpeg_enc_frame* __restrict__ frames,
            const x3d_jpeg_enc_tables* __restrict__ tables, const int64_t* __restrict__ boff,
            const x3d_jpeg_enc_result* __restrict__ res, uint32_t* __restrict__ words) {
  __shared__ EncSmem sm;
  const x3d_jpeg_enc_frame fr = frames[blockIdx.y];
  const Grid g(fr);
  const int s0 = blockIdx.x * kEmitThreads;
  if (s0 >= g.nblocks || res[blockIdx.y].status != X3D_JPEG_OK) return;
  load_tables(sm, tables[fr.tables]);
  __syncthreads();
  const int s = s0 + threadIdx.x;
  if (s >= g.nblocks) return;
  const int16_t* cf = coef + fr.coef_off * 64;
  int c;
  const int b = g.block(s, c), p = g.prev_block(s);
  const int64_t pos = boff[fr.coef_off + s];
  WordWriter ww{words + fr.word_off + (pos >> 5), 0ull, static_cast<int>(pos & 31), 0};
  encode_block(cf + static_cast<int64_t>(b) * 64, p < 0 ? 0 : cf[static_cast<int64_t>(p) * 64], c, sm,
               [&](uint32_t code, int l) { ww.put(code, l); });
  if (s == g.nblocks - 1) {
    const int pad = static_cast<int>((8 - (res[blockIdx.y].bits & 7)) & 7);      // flush_bits
    if (pad) ww.put((1u << pad) - 1u, pad);
  }
  ww.finish();
}

// Stage C2, first launch: one CTA scans the frames' bound on their stuffed length, 2 x the unstuffed
// bytes, into res[f].out_off (an exclusive scan over the batch, O(nframes)).
constexpr int kOffsetThreads = 1024;

__global__ void __launch_bounds__(kOffsetThreads)
offsets_kernel(x3d_jpeg_enc_result* __restrict__ res, int nframes) {
  using Scan = cub::BlockScan<int64_t, kOffsetThreads>;
  __shared__ typename Scan::TempStorage tmp;
  __shared__ int64_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int f0 = 0; f0 < nframes; f0 += kOffsetThreads) {
    const int f = f0 + threadIdx.x;
    const int64_t bound = f < nframes ? 2 * ((res[f].bits + 7) >> 3) : 0;
    int64_t excl, total;
    Scan(tmp).ExclusiveSum(bound, excl, total);
    const int64_t base = carry;
    if (f < nframes) res[f].out_off = base + excl;
    __syncthreads();
    if (threadIdx.x == 0) carry = base + total;
    __syncthreads();
  }
}

// Stage C2, second launch: one CTA per frame stuffs a 0x00 after every 0xFF byte of the padded
// stream, a word per thread and step, into `out` at res[f].out_off.
constexpr int kStuffThreads = 512;

__global__ void __launch_bounds__(kStuffThreads)
stuff_kernel(const uint32_t* __restrict__ words, const x3d_jpeg_enc_frame* __restrict__ frames,
             x3d_jpeg_enc_result* __restrict__ res, uint8_t* __restrict__ out, int64_t out_cap) {
  using Scan = cub::BlockScan<int, kStuffThreads>;
  __shared__ typename Scan::TempStorage tmp;
  __shared__ int64_t carry;
  const int f = blockIdx.x;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int64_t o = res[f].out_off;
  const int64_t nbytes = (res[f].bits + 7) >> 3;
  if (res[f].status != X3D_JPEG_OK) return;
  if (o + 2 * nbytes > out_cap) {
    if (threadIdx.x == 0) res[f].status = X3D_JPEG_OVERFLOW;
    return;
  }
  const uint32_t* w = words + frames[f].word_off;
  const int64_t nw = (nbytes + 3) >> 2;
  for (int64_t i0 = 0; i0 < nw; i0 += kStuffThreads) {
    const int64_t i = i0 + threadIdx.x;
    const uint32_t word = i < nw ? w[i] : 0u;
    const int nb = i < nw ? static_cast<int>(nbytes - 4 * i < 4 ? nbytes - 4 * i : 4) : 0;
    int ff = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) ff += k < nb && ((word >> (24 - 8 * k)) & 0xFF) == 0xFF;
    int excl, total;
    Scan(tmp).ExclusiveSum(ff, excl, total);
    uint8_t* dst = out + o + carry + 4 * i + excl;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (k < nb) {
        const uint8_t v = static_cast<uint8_t>(word >> (24 - 8 * k));
        *dst++ = v;
        if (v == 0xFF) *dst++ = 0;
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) res[f].len = nbytes + carry;
}

}  // namespace jpeg_enc
}  // namespace x3d

using namespace x3d;

static bool aligned(const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

extern "C" int x3d_jpeg_fdct(const uint8_t* rgb, const x3d_jpeg_enc_frame* frames, const x3d_jpeg_enc_tables* tables,
                             int nframes, int max_blocks, int16_t* coef, void* stream) {
  X3D_REQUIRE(rgb && frames && tables && coef, X3D_ERR_INVALID_ARG, "x3d_jpeg_fdct: null pointer");
  X3D_REQUIRE(nframes > 0 && nframes <= 65535 && max_blocks > 0, X3D_ERR_INVALID_ARG,
              "x3d_jpeg_fdct: nframes=%d (1..65535) max_blocks=%d", nframes, max_blocks);
  X3D_REQUIRE(aligned(coef, 16) && aligned(frames, 8) && aligned(tables, 2), X3D_ERR_INVALID_ARG,
              "x3d_jpeg_fdct: coef must be 16-byte, frames 8-byte, tables 2-byte aligned");
  const dim3 grid((max_blocks + jpeg_enc::kFdctBlocks - 1) / jpeg_enc::kFdctBlocks, nframes);
  jpeg_enc::fdct_kernel<<<grid, jpeg_enc::kFdctBlocks * 8, 0, static_cast<cudaStream_t>(stream)>>>(rgb, frames, tables, coef);
  return check_launch("x3d_jpeg_fdct");
}

extern "C" int x3d_jpeg_enc_bits(const int16_t* coef, const x3d_jpeg_enc_frame* frames, const x3d_jpeg_enc_tables* tables,
                                 int nframes, int64_t* boff, x3d_jpeg_enc_result* res, uint32_t* words, void* stream) {
  X3D_REQUIRE(coef && frames && tables && boff && res && words, X3D_ERR_INVALID_ARG, "x3d_jpeg_enc_bits: null pointer");
  X3D_REQUIRE(nframes > 0, X3D_ERR_INVALID_ARG, "x3d_jpeg_enc_bits: nframes=%d", nframes);
  X3D_REQUIRE(aligned(coef, 2) && aligned(frames, 8) && aligned(tables, 2) && aligned(boff, 8) && aligned(res, 8) &&
              aligned(words, 4), X3D_ERR_INVALID_ARG,
              "x3d_jpeg_enc_bits: frames/boff/res must be 8-byte, words 4-byte, coef/tables 2-byte aligned");
  jpeg_enc::bits_kernel<<<nframes, jpeg_enc::kEncThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      coef, frames, tables, boff, res, words);
  return check_launch("x3d_jpeg_enc_bits");
}

extern "C" int x3d_jpeg_enc_emit(const int16_t* coef, const x3d_jpeg_enc_frame* frames, const x3d_jpeg_enc_tables* tables,
                                 int nframes, int max_blocks, const int64_t* boff, const x3d_jpeg_enc_result* res,
                                 uint32_t* words, void* stream) {
  X3D_REQUIRE(coef && frames && tables && boff && res && words, X3D_ERR_INVALID_ARG, "x3d_jpeg_enc_emit: null pointer");
  X3D_REQUIRE(nframes > 0 && nframes <= 65535 && max_blocks > 0, X3D_ERR_INVALID_ARG,
              "x3d_jpeg_enc_emit: nframes=%d (1..65535) max_blocks=%d", nframes, max_blocks);
  X3D_REQUIRE(aligned(coef, 2) && aligned(frames, 8) && aligned(tables, 2) && aligned(boff, 8) && aligned(res, 8) &&
              aligned(words, 4), X3D_ERR_INVALID_ARG,
              "x3d_jpeg_enc_emit: frames/boff/res must be 8-byte, words 4-byte, coef/tables 2-byte aligned");
  const dim3 grid((max_blocks + jpeg_enc::kEmitThreads - 1) / jpeg_enc::kEmitThreads, nframes);
  jpeg_enc::emit_kernel<<<grid, jpeg_enc::kEmitThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      coef, frames, tables, boff, res, words);
  return check_launch("x3d_jpeg_enc_emit");
}

extern "C" int x3d_jpeg_enc_stuff(const uint32_t* words, const x3d_jpeg_enc_frame* frames, int nframes,
                                  x3d_jpeg_enc_result* res, uint8_t* out, int64_t out_cap, void* stream) {
  X3D_REQUIRE(words && frames && res && out, X3D_ERR_INVALID_ARG, "x3d_jpeg_enc_stuff: null pointer");
  X3D_REQUIRE(nframes > 0 && out_cap >= 0, X3D_ERR_INVALID_ARG, "x3d_jpeg_enc_stuff: nframes=%d out_cap=%lld",
              nframes, (long long)out_cap);
  X3D_REQUIRE(aligned(words, 4) && aligned(frames, 8) && aligned(res, 8), X3D_ERR_INVALID_ARG,
              "x3d_jpeg_enc_stuff: frames/res must be 8-byte, words 4-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  jpeg_enc::offsets_kernel<<<1, jpeg_enc::kOffsetThreads, 0, st>>>(res, nframes);
  jpeg_enc::stuff_kernel<<<nframes, jpeg_enc::kStuffThreads, 0, st>>>(words, frames, res, out, out_cap);
  return check_launch("x3d_jpeg_enc_stuff");
}
