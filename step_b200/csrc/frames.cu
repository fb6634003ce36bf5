// frames.cu -- the reference's test-time input transform (BaseTransform, data/augmentations.py:601-615, then the BGR -> RGB
// swap and permute of data/ava.py:330-338) on the device, from decoded uint8 BGR frames.
//
// Per output value, in the reference's order and fp32 rounding (compiled with -fmad=false; every product and sum below is
// an explicitly rounded intrinsic, so no contraction can change a result):
//   ConvertFromInts (augmentations.py:75-84)  scale 0: u,  1: u / 255,  2: u * 2 / 255 - 1      (a 256-entry table)
//   Resize (:162-169)  cv2.resize INTER_LINEAR on float32: horizontal blend of two source columns, rounded to fp32, then the
//                      vertical blend of two such rows; cv2's sample positions and weights (resize_tap), index and weight
//                      clamped at both borders
//   SubtractMeans / DivideStds  (v - mean[c]) / std[c] with c the BGR channel
// Both entries compute every value with frame_value(), so the s2d form equals step_clip_to_s2d_f16 applied to the clip form
// bit for bit.
#include "common.cuh"

namespace step {
namespace {

struct FrameNorm {
  float mean[3], std[3];   // BGR order, as BaseTransform receives them
  int scale;
  int identity;            // all means 0 and stds 1 (the I3D setting, config.py:126-129): (v - 0) / 1 == v exactly
};

// one tap pair of the linear resize along one axis: out = s[i0] * w0 + s[i1] * w1
struct Tap {
  int i0, i1;
  float w0, w1;
};

// cv2 resize coefficients (INTER_LINEAR): f = (d + 0.5) * src / dst - 0.5 in double, s = floor(f), weight (float)(f - s)
// (the fraction is taken in double, then rounded: the weights match cv2's exactly); left of the first source sample s = 0
// and weight 0, at or right of the last one s = src - 1 and weight 0.
__device__ __forceinline__ Tap resize_tap(int d, int src, int dst) {
  const double fd = ((double)d + 0.5) * ((double)src / (double)dst) - 0.5;
  int s = (int)floor(fd);
  float f = (float)(fd - (double)s);
  if (s < 0) { s = 0; f = 0.0f; }
  if (s >= src - 1) { s = src - 1; f = 0.0f; }
  Tap t;
  t.i0 = s;
  t.i1 = min(s + 1, src - 1);
  t.w0 = __fsub_rn(1.0f, f);
  t.w1 = f;
  return t;
}

__device__ __forceinline__ float convert_from_int(int u, int scale) {
  const float f = (float)u;
  if (scale == 0) return f;
  if (scale == 1) return __fdiv_rn(f, 255.0f);
  return __fsub_rn(__fdiv_rn(__fmul_rn(f, 2.0f), 255.0f), 1.0f);
}

// one output value of channel cb (BGR) at the sample taps (ty, tx) of a frame with row pitch `pitch` bytes
__device__ __forceinline__ float frame_value(const uint8_t* __restrict__ frame, size_t pitch, const Tap& ty, const Tap& tx,
                                             int cb, const float* __restrict__ tab, const FrameNorm& nm) {
  const uint8_t* r0 = frame + (size_t)ty.i0 * pitch + cb;
  const uint8_t* r1 = frame + (size_t)ty.i1 * pitch + cb;
  const float h0 = __fadd_rn(__fmul_rn(tab[__ldg(r0 + 3 * tx.i0)], tx.w0), __fmul_rn(tab[__ldg(r0 + 3 * tx.i1)], tx.w1));
  const float h1 = __fadd_rn(__fmul_rn(tab[__ldg(r1 + 3 * tx.i0)], tx.w0), __fmul_rn(tab[__ldg(r1 + 3 * tx.i1)], tx.w1));
  const float v = __fadd_rn(__fmul_rn(h0, ty.w0), __fmul_rn(h1, ty.w1));
  if (nm.identity) return v;
  return __fdiv_rn(__fsub_rn(v, nm.mean[cb]), nm.std[cb]);
}

// ConvertFromInts table in shared memory (blockDim.x >= 256)
__device__ __forceinline__ void fill_table(float* tab, int scale) {
  if (threadIdx.x < 256) tab[threadIdx.x] = convert_from_int(threadIdx.x, scale);
  __syncthreads();
}

// source extent of clip n from the device size table, clamped into the frame slot (the host validates it; the clamp only
// keeps a bad table from reading outside the batch)
__device__ __forceinline__ void clip_extent(const int32_t* __restrict__ sizes, int n, int Hmax, int Wmax, int& H0, int& W0) {
  H0 = min(max(__ldg(sizes + 2 * n), 1), Hmax);
  W0 = min(max(__ldg(sizes + 2 * n + 1), 1), Wmax);
}

// [N,T,Hmax,Wmax,3] u8 -> [N,T,3,H,W] fp32 RGB; one thread per output pixel (three planes)
__global__ void __launch_bounds__(256) frames_to_clip_kernel(const uint8_t* __restrict__ frames, const int32_t* __restrict__ sizes,
                                                             int T_, int Hmax, int Wmax, int H, int W, long long total, FrameNorm nm,
                                                             float* __restrict__ out) {
  __shared__ float tab[256];
  fill_table(tab, nm.scale);
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int x = (int)(idx % W);
  long long r = idx / W;
  const int y = (int)(r % H);
  const long long nt = r / H;
  const int n = (int)(nt / T_);
  int H0, W0;
  clip_extent(sizes, n, Hmax, Wmax, H0, W0);
  const size_t pitch = (size_t)Wmax * 3;
  const uint8_t* frame = frames + (size_t)nt * Hmax * pitch;
  const Tap ty = resize_tap(y, H0, H), tx = resize_tap(x, W0, W);
  float* o = out + (size_t)nt * 3 * H * W + (size_t)y * W + x;
#pragma unroll
  for (int c = 0; c < 3; ++c) o[(size_t)c * H * W] = frame_value(frame, pitch, ty, tx, 2 - c, tab, nm);
}

// [N,T,Hmax,Wmax,3] u8 -> s2d [N,T/2,H/2,W/2,32] f16, channel ((rt*2+rh)*2+rw)*3 + c (RGB), channels 24..31 zero: the layout of
// clip_to_s2d_rgb_kernel (pool_layout.cu).  One thread per output pixel: 24 values, two 32-byte stores.
__global__ void __launch_bounds__(256) frames_to_s2d_kernel(const uint8_t* __restrict__ frames, const int32_t* __restrict__ sizes,
                                                            int T_, int Hmax, int Wmax, int H, int W, long long total, FrameNorm nm,
                                                            __half* __restrict__ out) {
  __shared__ float tab[256];
  fill_table(tab, nm.scale);
  const int T2 = T_ / 2, H2 = H / 2, W2 = W / 2;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int w2 = (int)(idx % W2);
  long long r = idx / W2;
  const int h2 = (int)(r % H2); r /= H2;
  const int t2 = (int)(r % T2);
  const int n = (int)(r / T2);
  int H0, W0;
  clip_extent(sizes, n, Hmax, Wmax, H0, W0);
  const size_t pitch = (size_t)Wmax * 3;
  Tap tx[2], ty[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    tx[k] = resize_tap(2 * w2 + k, W0, W);
    ty[k] = resize_tap(2 * h2 + k, H0, H);
  }
  float v[32];
#pragma unroll
  for (int k = 24; k < 32; ++k) v[k] = 0.0f;
#pragma unroll
  for (int rt = 0; rt < 2; ++rt) {
    const uint8_t* frame = frames + ((size_t)n * T_ + 2 * t2 + rt) * Hmax * pitch;
#pragma unroll
    for (int rh = 0; rh < 2; ++rh)
#pragma unroll
      for (int rw = 0; rw < 2; ++rw)
#pragma unroll
        for (int c = 0; c < 3; ++c)
          v[((rt * 2 + rh) * 2 + rw) * 3 + c] = frame_value(frame, pitch, ty[rh], tx[rw], 2 - c, tab, nm);
  }
  uint32_t o[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const __half2 h = __floats2half2_rn(v[2 * k], v[2 * k + 1]);
    o[k] = *reinterpret_cast<const uint32_t*>(&h);
  }
  __half* dst = out + (size_t)idx * 32;
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]),
               "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst + 16), "r"(o[8]), "r"(o[9]), "r"(o[10]), "r"(o[11]),
               "r"(o[12]), "r"(o[13]), "r"(o[14]), "r"(o[15]) : "memory");
}

// host-side argument checks shared by both entries; fills nm
int check_frames_args(const char* name, const uint8_t* frames, const int32_t* sizes, int N, int T, int Hmax, int Wmax, int H, int W,
                      int scale, const float* mean, const float* stds, const void* out, FrameNorm& nm) {
  STEP_CHECK_ARG(frames && sizes && out, "%s: null pointer", name);
  STEP_CHECK_ARG(N > 0 && T > 0 && Hmax > 0 && Wmax > 0 && H > 0 && W > 0, "%s: bad extent N=%d T=%d Hmax=%d Wmax=%d H=%d W=%d",
                 name, N, T, Hmax, Wmax, H, W);
  STEP_CHECK_ARG((long long)Hmax * Wmax * 3 <= 0x7fffffffLL, "%s: frame slot %d x %d x 3 exceeds 2^31 bytes", name, Hmax, Wmax);
  STEP_CHECK_ARG((long long)N * T * H * W <= (1LL << 40), "%s: output too large", name);
  STEP_CHECK_ARG(scale == 0 || scale == 1 || scale == 2, "%s: scale must be 0, 1 or 2 (got %d)", name, scale);
  STEP_CHECK_ARG(((uintptr_t)sizes & 3) == 0, "%s: sizes must be 4-byte aligned", name);
  for (int c = 0; c < 3; ++c) {
    STEP_CHECK_ARG(stds[c] != 0.0f && isfinite(stds[c]) && isfinite(mean[c]), "%s: mean/std of channel %d must be finite, std non-zero",
                   name, c);
    nm.mean[c] = mean[c];
    nm.std[c] = stds[c];
  }
  nm.scale = scale;
  nm.identity = mean[0] == 0.0f && mean[1] == 0.0f && mean[2] == 0.0f && stds[0] == 1.0f && stds[1] == 1.0f && stds[2] == 1.0f;
  return 0;
}

}  // namespace
}  // namespace step

using namespace step;

extern "C" int step_frames_to_clip_f32(const uint8_t* frames, const int32_t* sizes, int N, int T, int Hmax, int Wmax, int H, int W,
                                       int scale, float mean_b, float mean_g, float mean_r, float std_b, float std_g, float std_r,
                                       float* out, step_stream_t stream) {
  const float mean[3] = {mean_b, mean_g, mean_r}, stds[3] = {std_b, std_g, std_r};
  FrameNorm nm;
  if (int rc = check_frames_args("frames_to_clip", frames, sizes, N, T, Hmax, Wmax, H, W, scale, mean, stds, out, nm)) return rc;
  STEP_CHECK_ARG(((uintptr_t)out & 3) == 0, "frames_to_clip: out must be 4-byte aligned");
  const long long total = (long long)N * T * H * W;
  STEP_CHECK_ARG(ceil_div(total, 256) < (1LL << 31), "frames_to_clip: too many pixels");
  frames_to_clip_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, cu(stream)>>>(frames, sizes, T, Hmax, Wmax, H, W, total, nm, out);
  STEP_LAUNCH_CHECK("frames_to_clip_kernel");
  return 0;
}

extern "C" int step_frames_to_s2d_f16(const uint8_t* frames, const int32_t* sizes, int N, int T, int Hmax, int Wmax, int H, int W,
                                      int scale, float mean_b, float mean_g, float mean_r, float std_b, float std_g, float std_r,
                                      void* out, step_stream_t stream) {
  const float mean[3] = {mean_b, mean_g, mean_r}, stds[3] = {std_b, std_g, std_r};
  FrameNorm nm;
  if (int rc = check_frames_args("frames_to_s2d", frames, sizes, N, T, Hmax, Wmax, H, W, scale, mean, stds, out, nm)) return rc;
  STEP_CHECK_ARG(T % 2 == 0 && H % 2 == 0 && W % 2 == 0, "frames_to_s2d: T, H, W must be even (T=%d H=%d W=%d)", T, H, W);
  STEP_CHECK_ARG(((uintptr_t)out & 31) == 0, "frames_to_s2d: out must be 32-byte aligned");
  const long long total = (long long)N * (T / 2) * (H / 2) * (W / 2);
  STEP_CHECK_ARG(ceil_div(total, 256) < (1LL << 31), "frames_to_s2d: too many pixels");
  frames_to_s2d_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, cu(stream)>>>(frames, sizes, T, Hmax, Wmax, H, W, total, nm,
                                                                               (__half*)out);
  STEP_LAUNCH_CHECK("frames_to_s2d_kernel");
  return 0;
}
