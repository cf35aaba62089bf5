// The two steps either side of the forward path that run on the device:
//   * input stage  -- utils.normalize (reference utils.py:42-72) on decoded uint8 frames;
//   * eval metrics -- the loss and metrics eval.py:62-70 compiles into the model
//     (SparseCategoricalCrossentropy on probabilities, SparseCategoricalAccuracy,
//     SparseTopKCategoricalAccuracy(k)).
#include "common.cuh"

namespace x3d {
namespace io {

struct Norm {
  float mean[3], std[3], nv;
};

// Same fp32 operation order as the reference: x / norm_value, then (x - mean) / std.
__device__ __forceinline__ float normalize1(float u, float nv, float mean, float std) {
  return __fdiv_rn(__fsub_rn(__fdiv_rn(u, nv), mean), std);
}

// A pixel value can only be one of 256 per channel, so every CTA first builds the 3 x 256 table of
// normalised values (exact IEEE fp32 in the reference's order, rounded once for bf16 output) in
// shared memory and the streaming loop is a byte extract + table read per element: 12 bytes in
// (three 32-bit loads = 4 pixels), 12 values out (16-byte stores) per thread and iteration.
template <typename TO>
__global__ void __launch_bounds__(256)
normalize_u8_kernel(const uint8_t* __restrict__ in, TO* __restrict__ out, int64_t pixels, const Norm nrm) {
  __shared__ TO lut[3][256];
  for (int i = threadIdx.x; i < 768; i += blockDim.x) {
    const int ch = i >> 8;
    const float r = normalize1(static_cast<float>(i & 255), nrm.nv, nrm.mean[ch], nrm.std[ch]);
    if (sizeof(TO) == 4) reinterpret_cast<float*>(&lut[0][0])[i] = r;
    else reinterpret_cast<bf16*>(&lut[0][0])[i] = __float2bfloat16_rn(r);
  }
  __syncthreads();
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const int64_t groups = pixels / 4;
  for (int64_t g = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; g < groups; g += stride) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(in + g * 12);
    const uint32_t w[3] = {__ldg(src), __ldg(src + 1), __ldg(src + 2)};
    TO v[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) v[i] = lut[i % 3][(w[i >> 2] >> (8 * (i & 3))) & 0xffu];
    if (sizeof(TO) == 4) {
      float4* dst = reinterpret_cast<float4*>(out + g * 12);
      const float* f = reinterpret_cast<const float*>(v);
#pragma unroll
      for (int i = 0; i < 3; ++i) dst[i] = make_float4(f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]);
    } else {
      // 24 bytes: 8-byte aligned for every g, 16-byte aligned for even g
      uint2* dst = reinterpret_cast<uint2*>(out + g * 12);
      const uint32_t* u = reinterpret_cast<const uint32_t*>(v);
#pragma unroll
      for (int i = 0; i < 3; ++i) dst[i] = make_uint2(u[2 * i], u[2 * i + 1]);
    }
  }
  // tail (pixels % 4) by the first threads of block 0
  if (blockIdx.x == 0) {
    const int64_t done = groups * 4;
    for (int64_t e = done * 3 + threadIdx.x; e < pixels * 3; e += blockDim.x) out[e] = lut[e % 3][in[e]];
  }
}

// One warp per video.  Keras semantics (TF 2.4 backend.sparse_categorical_crossentropy with
// from_logits=False on a tensor that is not a Softmax op output -- eval-mode X3D.call returns a
// mean over views): p = clip(p, 1e-7, 1 - 1e-7); loss = -(log p[label] - log sum_j p[j]).
// top-1: argmax (first maximal index) == label.  top-k: tf.math.in_top_k, i.e. fewer than k
// classes have a strictly larger probability.
__global__ void __launch_bounds__(128)
eval_metrics_kernel(const float* __restrict__ probs, const int32_t* __restrict__ labels,
                    double* __restrict__ acc, int V, int ncls, int k) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= V) return;
  const float* p = probs + static_cast<int64_t>(warp) * ncls;
  const int label = labels[warp];
  if (label < 0 || label >= ncls) return;                   // counted as a miss with zero loss
  const float pl = p[label];
  int greater = 0, before = 0;
  float sum = 0.f;
  for (int j = lane; j < ncls; j += 32) {
    const float v = p[j];
    greater += v > pl;
    before += (v == pl && j < label);
    sum += fminf(fmaxf(v, 1e-7f), 1.f - 1e-7f);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    greater += __shfl_xor_sync(0xffffffffu, greater, o);
    before += __shfl_xor_sync(0xffffffffu, before, o);
    sum += __shfl_xor_sync(0xffffffffu, sum, o);
  }
  if (lane == 0) {
    const float plc = fminf(fmaxf(pl, 1e-7f), 1.f - 1e-7f);
    atomicAdd(acc + 0, static_cast<double>(logf(sum) - logf(plc)));
    atomicAdd(acc + 1, (greater == 0 && before == 0) ? 1.0 : 0.0);
    atomicAdd(acc + 2, greater < k ? 1.0 : 0.0);
    atomicAdd(acc + 3, 1.0);
  }
}

// Clips of decoded videos at any resolution: per output frame, a bilinear short-side resize
// (TF 2.4 ResizeBilinear, half_pixel_centers=True, what tf.image.resize(method="bilinear") runs,
// then tf.cast to uint8), a crop and an optional left-right flip, as ONE pass over the output.
//   out[n][t][y][x][c] = resize(frame(n, t), rh, rw)[y0 + y][x0 + (flip ? S-1-x : x)][c]
// The resized frame is never materialised: each output byte is interpolated from the four source
// bytes around its resized position.  fp32 arithmetic with every operation rounded on its own
// (__fmul_rn / __fadd_rn / __fsub_rn, which nvcc never contracts into an FMA):
//   scale = H / rh;  in = (y + 0.5) * scale - 0.5;  lo = max(floor(in), 0);  hi = min(ceil(in), H-1)
//   l = in - floor(in);  top = tl + (tr - tl) * lx;  bot = bl + (br - bl) * lx;  v = top + (bot - top) * ly
//   out = trunc(v)
// A CTA owns kRows output rows of one output frame.  It first tabulates the source column byte
// offsets and weights of all S output columns of its clip (and the source rows of its kRows rows) in
// shared memory; then each thread produces 4 output pixels (12 bytes) per item, stored as three
// 32-bit words when the row starts 4-byte aligned (S % 4 == 0), byte by byte otherwise.
//
// The per-clip plan (source frame of every output frame, x3d_clip_desc) comes from one of two
// sources: device arrays (x3d_video_clips_u8) or, for x3d_eval_views_u8, values passed by argument
// (one video, identity resize, frame index computed from the view and time step).
constexpr int kRows = 16;
constexpr int kThreads = 256;
constexpr int kMaxS = 2048;

struct DescPlan {
  const int64_t* frame_off;
  const x3d_clip_desc* desc;
  __device__ __forceinline__ x3d_clip_desc clip(int n) const { return desc[n]; }
  __device__ __forceinline__ int64_t frame(int n, int t, int T) const { return frame_off[static_cast<int64_t>(n) * T + t]; }
};

struct ViewsPlan {
  x3d_clip_desc crop[3];
  int views, F, rate;
  int64_t frame_bytes;
  __device__ __forceinline__ x3d_clip_desc clip(int n) const {      // selects, not a dynamic index (no stack copy)
    const int i = n / views;
    return i == 0 ? crop[0] : (i == 1 ? crop[1] : crop[2]);
  }
  __device__ __forceinline__ int64_t frame(int n, int t, int T) const {
    const int64_t f = (static_cast<int64_t>(n % views) * T + t) * rate % F;
    return f * frame_bytes;
  }
};

// source position of output coordinate `o` along an axis resized from `in` to `out` samples
__device__ __forceinline__ void src_coord(int o, int in, int out, int& lo, int& hi, float& l) {
  const float scale = __fdiv_rn(static_cast<float>(in), static_cast<float>(out));
  const float p = __fsub_rn(__fmul_rn(__fadd_rn(static_cast<float>(o), 0.5f), scale), 0.5f);
  const float fl = floorf(p);
  lo = max(static_cast<int>(fl), 0);
  hi = min(static_cast<int>(ceilf(p)), in - 1);
  lo = min(lo, in - 1);
  l = __fsub_rn(p, fl);
}

__device__ __forceinline__ uint32_t lerp_u8(uint32_t tl, uint32_t tr, uint32_t bl, uint32_t br, float lx, float ly) {
  const float ftl = static_cast<float>(tl), fbl = static_cast<float>(bl);
  const float top = __fadd_rn(ftl, __fmul_rn(__fsub_rn(static_cast<float>(tr), ftl), lx));
  const float bot = __fadd_rn(fbl, __fmul_rn(__fsub_rn(static_cast<float>(br), fbl), lx));
  const float v = __fadd_rn(top, __fmul_rn(__fsub_rn(bot, top), ly));
  return static_cast<uint32_t>(v);                                   // truncation, as tf.cast
}

template <class Plan>
__global__ void __launch_bounds__(kThreads)
video_clips_u8_kernel(const uint8_t* __restrict__ frames, uint8_t* __restrict__ out, const Plan plan,
                      int T, int S, int bands) {
  extern __shared__ int32_t smem[];
  int32_t* xlo = smem;                       // [S] source byte offset within a row (column * 3)
  int32_t* xhi = xlo + S;
  float* lxs = reinterpret_cast<float*>(xhi + S);
  int32_t* ylo = reinterpret_cast<int32_t*>(lxs + S);   // [kRows] source row byte offset
  int32_t* yhi = ylo + kRows;
  float* lys = reinterpret_cast<float*>(yhi + kRows);

  const int64_t nt = blockIdx.x / bands;                 // output frame n*T + t
  const int band = static_cast<int>(blockIdx.x - nt * bands);
  const int n = static_cast<int>(nt / T), t = static_cast<int>(nt - static_cast<int64_t>(n) * T);
  const x3d_clip_desc d = plan.clip(n);
  const int row_bytes = d.W * 3;
  for (int x = threadIdx.x; x < S; x += blockDim.x) {
    const int rx = d.x0 + (d.flip ? S - 1 - x : x);
    int lo, hi; float l;
    src_coord(rx, d.W, d.rw, lo, hi, l);
    xlo[x] = lo * 3; xhi[x] = hi * 3; lxs[x] = l;
  }
  const int y_begin = band * kRows;
  const int rows = min(kRows, S - y_begin);
  if (threadIdx.x < rows) {
    int lo, hi; float l;
    src_coord(d.y0 + y_begin + threadIdx.x, d.H, d.rh, lo, hi, l);
    ylo[threadIdx.x] = lo * row_bytes; yhi[threadIdx.x] = hi * row_bytes; lys[threadIdx.x] = l;
  }
  __syncthreads();

  const uint8_t* src = frames + plan.frame(n, t, T);
  uint8_t* dst = out + (nt * S + y_begin) * static_cast<int64_t>(S) * 3;
  const int quads = (S + 3) >> 2;
  const bool wide = (S & 3) == 0;
  for (int item = threadIdx.x; item < rows * quads; item += blockDim.x) {
    const int r = item / quads, x0 = (item - r * quads) * 4;
    const uint8_t* top = src + ylo[r];
    const uint8_t* bot = src + yhi[r];
    const float ly = lys[r];
    uint32_t v[12];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const int x = min(x0 + p, S - 1);                  // the last quad of a row may be partial
      const int a = xlo[x], b = xhi[x];
      const float lx = lxs[x];
#pragma unroll
      for (int c = 0; c < 3; ++c)
        v[p * 3 + c] = lerp_u8(__ldg(top + a + c), __ldg(top + b + c), __ldg(bot + a + c), __ldg(bot + b + c), lx, ly);
    }
    uint8_t* o = dst + (static_cast<int64_t>(r) * S + x0) * 3;
    if (wide) {
      uint32_t* o32 = reinterpret_cast<uint32_t*>(o);
#pragma unroll
      for (int w = 0; w < 3; ++w)
        o32[w] = v[4 * w] | (v[4 * w + 1] << 8) | (v[4 * w + 2] << 16) | (v[4 * w + 3] << 24);
    } else {
      const int nb = min(4, S - x0) * 3;
      for (int b = 0; b < nb; ++b) o[b] = static_cast<uint8_t>(v[b]);
    }
  }
}

template <class Plan>
int launch_clips(const uint8_t* frames, uint8_t* out, const Plan& plan, int N, int T, int S, void* stream,
                 const char* what) {
  const int bands = (S + kRows - 1) / kRows;
  const int64_t blocks = static_cast<int64_t>(N) * T * bands;
  X3D_REQUIRE(blocks <= 0x7fffffffLL, X3D_ERR_UNSUPPORTED, "%s: %lld CTAs", what, (long long)blocks);
  const size_t smem = static_cast<size_t>(S) * 12 + kRows * 12;
  video_clips_u8_kernel<Plan><<<static_cast<unsigned>(blocks), kThreads, smem, static_cast<cudaStream_t>(stream)>>>(
      frames, out, plan, T, S, bands);
  return check_launch(what);
}

}  // namespace io
}  // namespace x3d

using namespace x3d;

// The same kernel over a plan that is not device data: one already resized video (identity resize,
// rh = H, rw = W), temporal views (transforms.py:48-65) and uniform crops (transforms.py:149-190,
// 216-222): centre = ceil((dim - S) / 2); with three crops the longer side gets 0 / centre / dim - S.
extern "C" int x3d_eval_views_u8(const uint8_t* video, uint8_t* out, int F, int H, int W, int T, int views,
                                 int crops, int S, void* stream) {
  X3D_REQUIRE(video && out, X3D_ERR_INVALID_ARG, "x3d_eval_views_u8: null pointer");
  X3D_REQUIRE(F > 0 && T > 0 && views > 0 && S > 0 && H >= S && W >= S, X3D_ERR_INVALID_ARG,
              "x3d_eval_views_u8: bad extents F=%d T=%d views=%d S=%d H=%d W=%d", F, T, views, S, H, W);
  X3D_REQUIRE(crops == 1 || crops == 3, X3D_ERR_INVALID_ARG, "x3d_eval_views_u8: crops=%d (1 or 3)", crops);
  X3D_REQUIRE(S <= io::kMaxS, X3D_ERR_UNSUPPORTED, "x3d_eval_views_u8: S=%d > %d", S, io::kMaxS);
  X3D_REQUIRE((reinterpret_cast<uintptr_t>(out) & 3) == 0, X3D_ERR_INVALID_ARG, "x3d_eval_views_u8: out must be 4-byte aligned");
  io::ViewsPlan p;
  p.views = views; p.F = F;
  p.rate = F / T > 1 ? F / T : 1;
  p.frame_bytes = static_cast<int64_t>(H) * W * 3;
  const int yc = (H - S + 1) / 2, xc = (W - S + 1) / 2;                // ceil((dim - S) / 2)
  for (int i = 0; i < 3; ++i) {
    const int idx = crops > 1 ? i % 3 : 1;                             // left/centre/right vs centre
    x3d_clip_desc& d = p.crop[i];
    d.H = H; d.W = W; d.rh = H; d.rw = W; d.flip = 0;
    d.y0 = yc; d.x0 = xc;
    if (H > W) { if (idx == 0) d.y0 = 0; else if (idx == 2) d.y0 = H - S; }
    else       { if (idx == 0) d.x0 = 0; else if (idx == 2) d.x0 = W - S; }
  }
  return io::launch_clips(video, out, p, crops * views, T, S, stream, "x3d_eval_views_u8");
}

extern "C" int x3d_video_clips_u8(const uint8_t* frames, const int64_t* frame_off, const x3d_clip_desc* desc,
                                  int N, int T, int S, uint8_t* out, void* stream) {
  X3D_REQUIRE(frames && frame_off && desc && out, X3D_ERR_INVALID_ARG, "x3d_video_clips_u8: null pointer");
  X3D_REQUIRE(N > 0 && T > 0 && S > 0, X3D_ERR_INVALID_ARG, "x3d_video_clips_u8: N=%d T=%d S=%d", N, T, S);
  X3D_REQUIRE(S <= io::kMaxS, X3D_ERR_UNSUPPORTED, "x3d_video_clips_u8: S=%d > %d", S, io::kMaxS);
  X3D_REQUIRE((reinterpret_cast<uintptr_t>(out) & 3) == 0 && (reinterpret_cast<uintptr_t>(frame_off) & 7) == 0 &&
              (reinterpret_cast<uintptr_t>(desc) & 3) == 0, X3D_ERR_INVALID_ARG,
              "x3d_video_clips_u8: out and desc must be 4-byte, frame_off 8-byte aligned");
  io::DescPlan p;
  p.frame_off = frame_off; p.desc = desc;
  return io::launch_clips(frames, out, p, N, T, S, stream, "x3d_video_clips_u8");
}

extern "C" int x3d_normalize_u8(const uint8_t* in, void* out, int64_t pixels, const float* mean,
                                const float* std, float norm_value, int dtype, void* stream) {
  X3D_REQUIRE(in && out && mean && std, X3D_ERR_INVALID_ARG, "x3d_normalize_u8: null pointer");
  X3D_REQUIRE(pixels > 0, X3D_ERR_INVALID_ARG, "x3d_normalize_u8: pixels=%lld", (long long)pixels);
  X3D_REQUIRE(dtype == X3D_F32 || dtype == X3D_BF16, X3D_ERR_INVALID_ARG, "x3d_normalize_u8: dtype %d", dtype);
  X3D_REQUIRE(norm_value != 0.f && std[0] != 0.f && std[1] != 0.f && std[2] != 0.f, X3D_ERR_INVALID_ARG,
              "x3d_normalize_u8: zero divisor");
  X3D_REQUIRE((reinterpret_cast<uintptr_t>(in) & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
              X3D_ERR_INVALID_ARG, "x3d_normalize_u8: in must be 4-byte, out 16-byte aligned");
  io::Norm nrm;
  for (int i = 0; i < 3; ++i) { nrm.mean[i] = mean[i]; nrm.std[i] = std[i]; }
  nrm.nv = norm_value;
  const int64_t groups = (pixels + 3) / 4;
  int64_t blocks = (groups + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == X3D_F32)
    io::normalize_u8_kernel<float><<<(int)blocks, 256, 0, st>>>(in, static_cast<float*>(out), pixels, nrm);
  else
    io::normalize_u8_kernel<bf16><<<(int)blocks, 256, 0, st>>>(in, static_cast<bf16*>(out), pixels, nrm);
  return check_launch("x3d_normalize_u8");
}

extern "C" int x3d_eval_metrics(const float* probs, const int32_t* labels, double* acc, int V, int ncls,
                                int k, void* stream) {
  X3D_REQUIRE(probs && labels && acc, X3D_ERR_INVALID_ARG, "x3d_eval_metrics: null pointer");
  X3D_REQUIRE(V > 0 && ncls > 0 && k > 0, X3D_ERR_INVALID_ARG, "x3d_eval_metrics: V=%d ncls=%d k=%d", V, ncls, k);
  const int blocks = (V + 3) / 4;
  io::eval_metrics_kernel<<<blocks, 128, 0, static_cast<cudaStream_t>(stream)>>>(probs, labels, acc, V, ncls, k);
  return check_launch("x3d_eval_metrics");
}
