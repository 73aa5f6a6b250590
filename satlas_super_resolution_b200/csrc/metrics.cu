// Validation metrics on the GPU (SURVEY.md 8f row 3): what nondist_validation of ssr/models/ssr_esrgan_model.py:269-352 computes per
// image on the host -- basicsr tensor2img, calculate_psnr / calculate_ssim, and the 81-offset brute-force search of
// ssr/metrics/cpsnr.py:7-59 -- batched over the whole validation batch.  PSNR and cPSNR are reduced to EXACT integer sums on the
// device (differences of uint8 images), so the host's float64 formula reproduces the reference bit for bit up to its own rounding.
#include "common.cuh"

namespace ssr {

static int grid_for_m(long work_items, int threads) {
  long blocks = (work_items + threads - 1) / threads;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

// basicsr tensor2img(rgb2bgr, out_type=uint8, min_max=(0, 1)): clamp, * 255, round half to even (np.round), HWC, optional RGB -> BGR
__global__ void f32_nchw_to_u8_hwc_kernel(const float* __restrict__ src, uint8_t* __restrict__ dst, int B, int C, int H, int W, int reverse) {
  const long HW = (long)H * W;
  const long total = (long)B * HW * C;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const long pix = i / C;
    const long n = pix / HW, hw = pix - n * HW;
    const int cs = reverse ? C - 1 - c : c;
    float v = src[(n * C + cs) * HW + hw];
    v = fminf(fmaxf(v, 0.f), 1.f);
    dst[i] = (uint8_t)__float2int_rn(v * 255.0f);
  }
}

// For image n, offset o = (ro, co) in [0, M]^2 and channel ch, over the (h - 2cb - M) x (w - 2cb - M) crop:
//   d = a[y + ro, x + co] - b[y + M - ro, x + M - co]   (both after removing `cb` border pixels);  S1 = sum d,  S2 = sum d^2
// out[((n * (M+1)^2 + o) * C + ch) * 2 + {0, 1}] (int64).  M = 0: the plain PSNR sums.
__global__ void u8_shift_diff_sums_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, int H, int W, int C, int cb,
                                          int M, long long* __restrict__ out) {
  const int o = blockIdx.x, n = blockIdx.y;
  const int ro = o / (M + 1), co = o - ro * (M + 1);
  const int ch_ = H - 2 * cb - M, cw_ = W - 2 * cb - M;
  const uint8_t* pa = a + (long)n * H * W * C;
  const uint8_t* pb = b + (long)n * H * W * C;
  long long s1[4] = {0, 0, 0, 0}, s2[4] = {0, 0, 0, 0};
  for (int p = threadIdx.x; p < ch_ * cw_; p += blockDim.x) {
    const int y = p / cw_, x = p - y * cw_;
    const uint8_t* qa = pa + ((long)(y + cb + ro) * W + (x + cb + co)) * C;
    const uint8_t* qb = pb + ((long)(y + cb + M - ro) * W + (x + cb + M - co)) * C;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      if (c < C) {
        const int d = (int)qa[c] - (int)qb[c];
        s1[c] += d;
        s2[c] += (long long)(d * d);
      }
    }
  }
  // warp sums -> one 64-bit atomic per warp, channel and moment (the caller zeroes `out`; two's complement makes the unsigned add exact)
  const int lane = threadIdx.x & 31;
  unsigned long long* dst = reinterpret_cast<unsigned long long*>(out) + (((long)n * (M + 1) * (M + 1) + o) * C) * 2;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    if (c < C) {
      long long v1 = s1[c], v2 = s2[c];
      for (int off = 16; off; off >>= 1) {
        v1 += __shfl_xor_sync(0xffffffffu, v1, off);
        v2 += __shfl_xor_sync(0xffffffffu, v2, off);
      }
      if (lane == 0) {
        atomicAdd(dst + 2 * c, (unsigned long long)v1);
        atomicAdd(dst + 2 * c + 1, (unsigned long long)v2);
      }
    }
  }
}

// basicsr calculate_ssim / _ssim: 11 x 11 Gaussian window (sigma 1.5) over the 'valid' region, per channel; out[n * C + c] += sum of
// the SSIM map (float64), the caller divides by the (h - 2cb - 10) * (w - 2cb - 10) map size.
__global__ void u8_ssim_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, int B, int H, int W, int C, int cb,
                               const double* __restrict__ win /* [11] */, double* __restrict__ out) {
  const int vh = H - 2 * cb - 10, vw = W - 2 * cb - 10;
  const long per = (long)vh * vw;
  const long total = (long)B * C * per;
  const double c1 = (0.01 * 255) * (0.01 * 255), c2 = (0.03 * 255) * (0.03 * 255);
  __shared__ double g[11];
  if (threadIdx.x < 11) g[threadIdx.x] = win[threadIdx.x];
  __syncthreads();
  for (long i0 = blockIdx.x * (long)blockDim.x; i0 < total; i0 += (long)gridDim.x * blockDim.x) {
    const long i = i0 + threadIdx.x;
    double val = 0.0;
    long key = -1;
    if (i < total) {
      const long nc = i / per, p = i - nc * per;
      const int n = (int)(nc / C), c = (int)(nc - (long)n * C);
      const int y = (int)(p / vw), x = (int)(p - (long)y * vw);
      const uint8_t* pa = a + ((long)n * H + y + cb) * W * C + (long)(x + cb) * C + c;
      const uint8_t* pb = b + ((long)n * H + y + cb) * W * C + (long)(x + cb) * C + c;
      double m1 = 0, m2 = 0, s11 = 0, s22 = 0, s12 = 0;
      for (int dy = 0; dy < 11; ++dy) {
        for (int dx = 0; dx < 11; ++dx) {
          const double wgt = g[dy] * g[dx];
          const double u = (double)pa[((long)dy * W + dx) * C], v = (double)pb[((long)dy * W + dx) * C];
          m1 += wgt * u;
          m2 += wgt * v;
          s11 += wgt * u * u;
          s22 += wgt * v * v;
          s12 += wgt * u * v;
        }
      }
      const double m11 = m1 * m1, m22 = m2 * m2, m12 = m1 * m2;
      val = ((2 * m12 + c1) * (2 * (s12 - m12) + c2)) / ((m11 + m22 + c1) * ((s11 - m11) + (s22 - m22) + c2));
      key = nc;
    }
    // consecutive threads mostly share (n, c): reduce the warp when they all do, else add one by one
    const long k0 = __shfl_sync(0xffffffffu, key, 0);
    const bool same = __all_sync(0xffffffffu, key == k0);
    if (same) {
      for (int off = 16; off; off >>= 1) val += __shfl_xor_sync(0xffffffffu, val, off);
      if ((threadIdx.x & 31) == 0 && key >= 0) atomicAdd(out + key, val);
    } else if (key >= 0) {
      atomicAdd(out + key, val);
    }
  }
}

// ------------------------------------------------------------------ LPIPS (lpips 0.1, net='vgg'; ssr/metrics/lpips.py:7-21)
// uint8 HWC image -> the 16-channel NHWC bf16 buffer conv1_1 reads: v = (x / 255 - shift[c]) / scale[c] (lpips ScalingLayer on the
// [0, 1] values calculate_lpips passes), channels [c, c_pad) zero.  One thread per pixel.
__global__ void ingest_u8_nhwc_kernel(const uint8_t* __restrict__ src, __nv_bfloat16* __restrict__ dst, long npix, int C, int dst_stride,
                                      int c_pad, const float* __restrict__ shift, const float* __restrict__ scale) {
  for (long p = blockIdx.x * (long)blockDim.x + threadIdx.x; p < npix; p += (long)gridDim.x * blockDim.x) {
    __nv_bfloat16* d = dst + p * dst_stride;
    for (int g = 0; g < c_pad; g += 8) {
      __align__(16) __nv_bfloat16 v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int c = g + j;
        float f = 0.f;
        if (c < C) f = ((float)src[p * C + c] / 255.f - shift[c]) / scale[c];
        v[j] = __float2bfloat16(f);
      }
      *reinterpret_cast<uint4*>(d + g) = *reinterpret_cast<const uint4*>(v);
    }
  }
}

__device__ __forceinline__ void bf16x8_to_f32(const uint4& v, float* f) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 t = __bfloat1622float2(h[j]);
    f[2 * j] = t.x;
    f[2 * j + 1] = t.y;
  }
}

constexpr int LPIPS_THREADS = 256;
constexpr int LPIPS_PIX_PER_CTA = 256;   // the partial-sum slots of an image depend on (h, w) only: batch-invariant by construction

// One tap of the LPIPS head.  x = [2b, h, w, C] post-ReLU features (images n and b + n are the pair); per pixel
//   d = sum_c lin[c] * (f0[c] / (|f0| + 1e-10) - f1[c] / (|f1| + 1e-10))^2
// with |f| = sqrt(sum_c f^2).  A group of LPP = min(32, C / 8) lanes owns one pixel, each lane VPL 16-byte vectors of both images held
// in registers; the two norms and d are butterfly sums over the group (every lane ends with the same bits).  CTA (t, n) covers pixels
// [t * 256, (t + 1) * 256) of pair n and writes their sum (fixed order, f64) to partial[n * gridDim.x + t].  No atomics.
template <int C>
__global__ void __launch_bounds__(LPIPS_THREADS) lpips_layer_sums_kernel(const __nv_bfloat16* __restrict__ x, int B, int hw,
                                                                         const float* __restrict__ lin, double* __restrict__ partial) {
  constexpr int LPP = C / 8 < 32 ? C / 8 : 32;
  constexpr int VPL = C / (8 * LPP);
  constexpr int GROUPS = LPIPS_THREADS / LPP;
  const int n = blockIdx.y;
  const int lane_g = threadIdx.x % LPP, grp = threadIdx.x / LPP;
  float w[VPL * 8];
#pragma unroll
  for (int v = 0; v < VPL; ++v) {
    const float4 a = *reinterpret_cast<const float4*>(lin + (v * LPP + lane_g) * 8);
    const float4 b = *reinterpret_cast<const float4*>(lin + (v * LPP + lane_g) * 8 + 4);
    w[v * 8 + 0] = a.x; w[v * 8 + 1] = a.y; w[v * 8 + 2] = a.z; w[v * 8 + 3] = a.w;
    w[v * 8 + 4] = b.x; w[v * 8 + 5] = b.y; w[v * 8 + 6] = b.z; w[v * 8 + 7] = b.w;
  }
  const __nv_bfloat16* x0 = x + (long)n * hw * C;
  const __nv_bfloat16* x1 = x + (long)(B + n) * hw * C;
  const int p_end = min(hw, (blockIdx.x + 1) * LPIPS_PIX_PER_CTA);
  float acc = 0.f;
  // the trip count is uniform over the CTA (the shuffles need whole warps); a group past the end reads zeros, which add 0
  for (int p0 = blockIdx.x * LPIPS_PIX_PER_CTA; p0 < p_end; p0 += GROUPS) {
    const int p = p0 + grp;
    float f0[VPL * 8], f1[VPL * 8];
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
      const long off = (long)p * C + (v * LPP + lane_g) * 8;
      const uint4 z = make_uint4(0u, 0u, 0u, 0u);
      bf16x8_to_f32(p < p_end ? *reinterpret_cast<const uint4*>(x0 + off) : z, f0 + v * 8);
      bf16x8_to_f32(p < p_end ? *reinterpret_cast<const uint4*>(x1 + off) : z, f1 + v * 8);
    }
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int j = 0; j < VPL * 8; ++j) {
      s0 = fmaf(f0[j], f0[j], s0);
      s1 = fmaf(f1[j], f1[j], s1);
    }
#pragma unroll
    for (int off = LPP / 2; off; off >>= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, off);
      s1 += __shfl_xor_sync(0xffffffffu, s1, off);
    }
    const float r0 = sqrtf(s0) + 1e-10f, r1 = sqrtf(s1) + 1e-10f;
    float d = 0.f;
#pragma unroll
    for (int j = 0; j < VPL * 8; ++j) {
      const float e = f0[j] / r0 - f1[j] / r1;
      d = fmaf(w[j], e * e, d);
    }
#pragma unroll
    for (int off = LPP / 2; off; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
    acc += d;
  }
  // the group's pixel sum -> shared memory, then one thread adds the groups in index order
  __shared__ double grp_sum[GROUPS];
  if (lane_g == 0) grp_sum[grp] = (double)acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int g = 0; g < GROUPS; ++g) s += grp_sum[g];
    partial[(long)n * gridDim.x + blockIdx.x] = s;
  }
}

struct LpipsTaps {
  int n_taps;
  int ctas[8];
  int hw[8];
  long offset[8];   // first partial of tap k (partials of tap k: [b][ctas[k]])
};

// out[n] = sum_k (sum_t partial_k[n][t]) / hw_k, every sum in f64 in index order
__global__ void lpips_finish_kernel(const double* __restrict__ partial, int B, LpipsTaps taps, double* __restrict__ out) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= B) return;
  double total = 0.0;
  for (int k = 0; k < taps.n_taps; ++k) {
    const double* p = partial + taps.offset[k] + (long)n * taps.ctas[k];
    double s = 0.0;
    for (int t = 0; t < taps.ctas[k]; ++t) s += p[t];
    total += s / (double)taps.hw[k];
  }
  out[n] = total;
}

}  // namespace ssr

using namespace ssr;
#define STREAM(s) reinterpret_cast<cudaStream_t>(s)

extern "C" int ssr_f32_nchw_to_u8_hwc(const float* src, void* dst_u8, int32_t b, int32_t c, int32_t h, int32_t w, int32_t reverse_channels,
                                      void* stream) {
  SSR_REQUIRE(src && dst_u8 && b > 0 && c > 0 && h > 0 && w > 0, "ssr_f32_nchw_to_u8_hwc: bad args");
  const long total = (long)b * c * h * w;
  f32_nchw_to_u8_hwc_kernel<<<grid_for_m(total, 256), 256, 0, STREAM(stream)>>>(src, reinterpret_cast<uint8_t*>(dst_u8), b, c, h, w,
                                                                               reverse_channels);
  count_launch();
  return check_last("f32_nchw_to_u8_hwc launch") ? SSR_OK : SSR_E_CUDA;
}

extern "C" int ssr_u8_shift_diff_sums(const void* a_u8, const void* b_u8, int32_t b, int32_t h, int32_t w, int32_t c, int32_t crop_border,
                                      int32_t max_offset, long long* out, void* stream) {
  SSR_REQUIRE(a_u8 && b_u8 && out && b > 0 && c > 0 && c <= 4, "ssr_u8_shift_diff_sums: bad args (1..4 channels)");
  SSR_REQUIRE(crop_border >= 0 && max_offset >= 0 && max_offset <= 16 && h - 2 * crop_border - max_offset > 0 && w - 2 * crop_border - max_offset > 0,
              "ssr_u8_shift_diff_sums: crop larger than the image");
  dim3 grid((unsigned)((max_offset + 1) * (max_offset + 1)), (unsigned)b);
  u8_shift_diff_sums_kernel<<<grid, 256, 0, STREAM(stream)>>>(reinterpret_cast<const uint8_t*>(a_u8), reinterpret_cast<const uint8_t*>(b_u8), h, w,
                                                            c, crop_border, max_offset, out);
  count_launch();
  return check_last("u8_shift_diff_sums launch") ? SSR_OK : SSR_E_CUDA;
}

extern "C" int ssr_u8_ssim_sums(const void* a_u8, const void* b_u8, int32_t b, int32_t h, int32_t w, int32_t c, int32_t crop_border,
                                const double* window11_device, double* out, void* stream) {
  SSR_REQUIRE(a_u8 && b_u8 && out && window11_device && b > 0 && c > 0, "ssr_u8_ssim_sums: bad args");
  SSR_REQUIRE(h - 2 * crop_border > 10 && w - 2 * crop_border > 10, "ssr_u8_ssim_sums: image smaller than the 11 x 11 window");
  const long total = (long)b * c * (h - 2 * crop_border - 10) * (w - 2 * crop_border - 10);
  u8_ssim_kernel<<<grid_for_m(total, 128), 128, 0, STREAM(stream)>>>(reinterpret_cast<const uint8_t*>(a_u8), reinterpret_cast<const uint8_t*>(b_u8),
                                                                    b, h, w, c, crop_border, window11_device, out);
  count_launch();
  return check_last("u8_ssim launch") ? SSR_OK : SSR_E_CUDA;
}

extern "C" int ssr_ingest_u8_nhwc(const void* src_u8, int32_t b, int32_t h, int32_t w, int32_t c, void* dst_bf16, int32_t dst_pix_stride,
                                  int32_t image_offset, int32_t c_pad, const float* shift, const float* scale, void* stream) {
  SSR_REQUIRE(src_u8 && dst_bf16 && shift && scale && b > 0 && h > 0 && w > 0 && c > 0 && image_offset >= 0, "ssr_ingest_u8_nhwc: bad args");
  SSR_REQUIRE(c_pad % 8 == 0 && c_pad >= c && dst_pix_stride % 8 == 0 && dst_pix_stride >= c_pad, "ssr_ingest_u8_nhwc: c_pad/stride");
  SSR_REQUIRE((reinterpret_cast<uintptr_t>(dst_bf16) & 15) == 0, "ssr_ingest_u8_nhwc: dst alignment");
  const long npix = (long)b * h * w;
  __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(dst_bf16) + (long)image_offset * h * w * dst_pix_stride;
  ingest_u8_nhwc_kernel<<<grid_for_m(npix, 256), 256, 0, STREAM(stream)>>>(reinterpret_cast<const uint8_t*>(src_u8), dst, npix, c, dst_pix_stride,
                                                                          c_pad, shift, scale);
  count_launch();
  return check_last("ingest_u8_nhwc launch") ? SSR_OK : SSR_E_CUDA;
}

extern "C" int32_t ssr_lpips_cta_count(int32_t h, int32_t w) {
  return (int32_t)((h * w + LPIPS_PIX_PER_CTA - 1) / LPIPS_PIX_PER_CTA);
}

extern "C" int ssr_lpips_layer_sums(const void* feat_bf16, int32_t b, int32_t h, int32_t w, int32_t c, const float* lin_w, double* partial,
                                    void* stream) {
  SSR_REQUIRE(feat_bf16 && lin_w && partial && b > 0 && h > 0 && w > 0, "ssr_lpips_layer_sums: bad args");
  SSR_REQUIRE((reinterpret_cast<uintptr_t>(feat_bf16) & 15) == 0 && (reinterpret_cast<uintptr_t>(lin_w) & 15) == 0,
              "ssr_lpips_layer_sums: alignment");
  SSR_REQUIRE(b <= 65535, "ssr_lpips_layer_sums: at most 65535 pairs");
  const dim3 grid((unsigned)ssr_lpips_cta_count(h, w), (unsigned)b);
  const __nv_bfloat16* x = reinterpret_cast<const __nv_bfloat16*>(feat_bf16);
  switch (c) {
    case 64: lpips_layer_sums_kernel<64><<<grid, LPIPS_THREADS, 0, STREAM(stream)>>>(x, b, h * w, lin_w, partial); break;
    case 128: lpips_layer_sums_kernel<128><<<grid, LPIPS_THREADS, 0, STREAM(stream)>>>(x, b, h * w, lin_w, partial); break;
    case 256: lpips_layer_sums_kernel<256><<<grid, LPIPS_THREADS, 0, STREAM(stream)>>>(x, b, h * w, lin_w, partial); break;
    case 512: lpips_layer_sums_kernel<512><<<grid, LPIPS_THREADS, 0, STREAM(stream)>>>(x, b, h * w, lin_w, partial); break;
    default: SSR_REQUIRE(false, "ssr_lpips_layer_sums: c must be 64, 128, 256 or 512 (got %d)", c);
  }
  count_launch();
  return check_last("lpips_layer_sums launch") ? SSR_OK : SSR_E_CUDA;
}

extern "C" int ssr_lpips_finish(const double* partial, int32_t b, int32_t n_taps, const int32_t* tap_h, const int32_t* tap_w, double* out,
                                void* stream) {
  SSR_REQUIRE(partial && out && tap_h && tap_w && b > 0 && n_taps > 0 && n_taps <= 8, "ssr_lpips_finish: bad args (1..8 taps)");
  LpipsTaps t;
  t.n_taps = n_taps;
  long off = 0;
  for (int k = 0; k < n_taps; ++k) {
    SSR_REQUIRE(tap_h[k] > 0 && tap_w[k] > 0, "ssr_lpips_finish: bad tap size");
    t.ctas[k] = ssr_lpips_cta_count(tap_h[k], tap_w[k]);
    t.hw[k] = tap_h[k] * tap_w[k];
    t.offset[k] = off;
    off += (long)b * t.ctas[k];
  }
  lpips_finish_kernel<<<(b + 127) / 128, 128, 0, STREAM(stream)>>>(partial, b, t, out);
  count_launch();
  return check_last("lpips_finish launch") ? SSR_OK : SSR_E_CUDA;
}
