// Small / bandwidth-bound kernels of the denoise step: small-M linear (time embeddings), sinusoidal embedding,
// nearest 2x upsample, channel concat, conv_in / conv_out (4-channel ends of the UNet, NCHW <-> NHWC), and the fused
// CFG-combine + Euler update + next-step input scaling (custom_pipelines.py:332-334,348-357).
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>

#include "../../include/ih_api.h"
#include "host_util.h"
#include "ptx.cuh"

namespace ih {

__device__ __forceinline__ void ld8(const __half* p, float (&x)[8]) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 f = unpack_half2(w[e]);
    x[2 * e] = f.x;
    x[2 * e + 1] = f.y;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// out[m, n] = act_out( W[n, :] . act_in(x[m, :]) + b[n] ),  M <= 8.  One warp per output column; W is read once.
// ---------------------------------------------------------------------------------------------------------------
constexpr int SL_MAXM = 8;
__global__ void linear_small_kernel(const __half* __restrict__ x, long long ldx, const __half* __restrict__ w,
                                    const __half* __restrict__ bias, const __half* __restrict__ addend,
                                    long long ld_add, __half* __restrict__ out, long long ldo, int M, int N, int K,
                                    int act_in, int act_out, float out_scale) {
  pdl_launch_dependents();
  pdl_wait();
  const int n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (n >= N) return;
  float acc[SL_MAXM];
#pragma unroll
  for (int m = 0; m < SL_MAXM; ++m) acc[m] = 0.f;
  const __half* wr = w + (long long)n * K;
  for (int k = lane * 8; k < K; k += 256) {
    float wv[8];
    ld8(wr + k, wv);
#pragma unroll
    for (int m = 0; m < SL_MAXM; ++m) {
      if (m < M) {
        float xv[8];
        ld8(x + m * ldx + k, xv);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float xe = xv[e];
          if (act_in == 1) xe = __half2float(__float2half_rn(silu_f(xe)));  // SiLU output is fp16 in the reference
          acc[m] += wv[e] * xe;
        }
      }
    }
  }
#pragma unroll
  for (int m = 0; m < SL_MAXM; ++m) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[m] += __shfl_xor_sync(0xffffffffu, acc[m], o);
  }
  if (lane == 0) {
    const float b = bias ? __half2float(bias[n]) : 0.f;
    for (int m = 0; m < M; ++m) {
      float y = __half2float(__float2half_rn(acc[m] + b));  // nn.Linear output is fp16 before the activation
      if (act_out == 1) y = silu_f(y);
      if (out_scale != 1.f) y = __half2float(__float2half_rn(y)) * out_scale;  // `module(x) * scale` on an fp16 tensor
      if (addend) y = __half2float(__float2half_rn(y)) + __half2float(addend[m * ld_add + n]);  // fp16 tensor add
      out[m * ldo + n] = __float2half_rn(y);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// sinusoid(t, dim) = [cos(t f_j), sin(t f_j)], f_j = exp(-ln(10000) j / half)   (flip_sin_to_cos=True, shift 0)
// ---------------------------------------------------------------------------------------------------------------
__global__ void sinusoid_kernel(const float* __restrict__ t, const int* __restrict__ step, __half* __restrict__ out,
                                long long ldo, int n, int dim) {
  pdl_launch_dependents();
  pdl_wait();
  const int half_dim = dim >> 1;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * half_dim) return;
  const int i = idx / half_dim, j = idx - i * half_dim;
  const float tv = step ? t[*step] : t[i];
  const float f = expf(-9.210340371976184f * (float)j / (float)half_dim);
  const float a = tv * f;
  out[i * ldo + j] = __float2half_rn(cosf(a));
  out[i * ldo + half_dim + j] = __float2half_rn(sinf(a));
}

__global__ void upsample2x_kernel(const uint4* __restrict__ x, uint4* __restrict__ out, int B, int H, int W, int CV) {
  pdl_launch_dependents();
  pdl_wait();
  const long long total = (long long)B * 2 * H * 2 * W * CV;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cv = (int)(i % CV);
    long long r = i / CV;
    const int ox = (int)(r % (2 * W));
    r /= (2 * W);
    const int oy = (int)(r % (2 * H));
    const int b = (int)(r / (2 * H));
    out[i] = x[(((long long)b * H + (oy >> 1)) * W + (ox >> 1)) * CV + cv];
  }
}

__global__ void concat_kernel(const uint4* __restrict__ x0, int CV0, const uint4* __restrict__ x1, int CV1,
                              uint4* __restrict__ out, long long rows) {
  pdl_launch_dependents();
  pdl_wait();
  const int CV = CV0 + CV1;
  const long long total = rows * CV;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cv = (int)(i % CV);
    const long long r = i / CV;
    out[i] = cv < CV0 ? x0[r * CV0 + cv] : x1[r * CV1 + (cv - CV0)];
  }
}

// ---------------------------------------------------------------------------------------------------------------
// conv_in: NCHW [B,Cin<=8,H,W] -> NHWC [B,H,W,Cout], 3x3 pad 1. thread = (pixel, 8 output channels)
// ---------------------------------------------------------------------------------------------------------------
__global__ void conv_in_kernel(const __half* __restrict__ x, const __half* __restrict__ w,
                               const __half* __restrict__ bias, __half* __restrict__ out, int B, int H, int W, int Cin,
                               int Cout) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ __half s_w[];  // [Cin*9][Cout]
  const int K = Cin * 9;
  for (int i = threadIdx.x; i < K * Cout; i += blockDim.x) {
    const int o = i / K, k = i - o * K;  // w is OIHW: [o][ci][ky][kx] -> k = ci*9 + ky*3 + kx
    s_w[k * Cout + o] = w[i];
  }
  __syncthreads();
  const int CG = Cout >> 3;
  const long long total = (long long)B * H * W * CG;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % CG);
    long long pix = i / CG;
    const int xw = (int)(pix % W);
    const int yh = (int)((pix / W) % H);
    const int b = (int)(pix / ((long long)W * H));
    float acc[8];
    if (bias) ld8(bias + cg * 8, acc);
    else {
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] = 0.f;
    }
    for (int ci = 0; ci < Cin; ++ci)
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const int yy = yh + t / 3 - 1, xx = xw + t % 3 - 1;
        if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
          const float xv = __half2float(x[(((long long)b * Cin + ci) * H + yy) * W + xx]);
          float wv[8];
          ld8(s_w + (ci * 9 + t) * Cout + cg * 8, wv);
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[e] += xv * wv[e];
        }
      }
    uint4 o;
    o.x = pack_half2(acc[0], acc[1]);
    o.y = pack_half2(acc[2], acc[3]);
    o.z = pack_half2(acc[4], acc[5]);
    o.w = pack_half2(acc[6], acc[7]);
    *reinterpret_cast<uint4*>(out + pix * Cout + cg * 8) = o;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// conv_out: NHWC [B,H,W,Cin] -> NCHW [B,Cout<=8,H,W], 3x3 pad 1. One warp per output pixel, lanes over channels.
// ---------------------------------------------------------------------------------------------------------------
constexpr int CO_MAX = 8;
__global__ void conv_out_kernel(const __half* __restrict__ x, const __half* __restrict__ w,
                                const __half* __restrict__ bias, __half* __restrict__ out, int B, int H, int W, int Cin,
                                int Cout) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ __half s_w[];  // [Cout][9][Cin]
  for (int i = threadIdx.x; i < Cout * 9 * Cin; i += blockDim.x) {
    const int o = i / (9 * Cin);
    const int rem = i - o * 9 * Cin;
    const int t = rem / Cin, ci = rem - t * Cin;
    s_w[i] = w[((long long)o * Cin + ci) * 9 + t];  // OIHW source
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  const long long npix = (long long)B * H * W;
  const int CV = Cin >> 3;
  for (long long pix = (long long)blockIdx.x * warps_per_block + (threadIdx.x >> 5); pix < npix;
       pix += (long long)gridDim.x * warps_per_block) {
    const int xw = (int)(pix % W);
    const int yh = (int)((pix / W) % H);
    const int b = (int)(pix / ((long long)W * H));
    float acc[CO_MAX];
#pragma unroll
    for (int o = 0; o < CO_MAX; ++o) acc[o] = 0.f;
    for (int t = 0; t < 9; ++t) {
      const int yy = yh + t / 3 - 1, xx = xw + t % 3 - 1;
      if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;  // warp-uniform
      const __half* src = x + (((long long)b * H + yy) * W + xx) * Cin;
      for (int cv = lane; cv < CV; cv += 32) {
        float xv[8];
        ld8(src + cv * 8, xv);
#pragma unroll
        for (int o = 0; o < CO_MAX; ++o) {
          if (o < Cout) {
            float wv[8];
            ld8(s_w + (o * 9 + t) * Cin + cv * 8, wv);
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[o] += xv[e] * wv[e];
          }
        }
      }
    }
#pragma unroll
    for (int o = 0; o < CO_MAX; ++o) {
#pragma unroll
      for (int s = 16; s > 0; s >>= 1) acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], s);
    }
    if (lane == 0) {
      for (int o = 0; o < Cout; ++o) {
        const float bv = bias ? __half2float(bias[o]) : 0.f;
        out[(((long long)b * Cout + o) * H + yh) * W + xw] = __float2half_rn(acc[o] + bv);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Inpainting blend, applied inside the Euler kernels (BLEND = true) after the update and before the next step's
// model_in is formed ([3P] diffusers StableDiffusionXLInpaintPipeline, 4-channel UNet, fp16 tensors):
//   proper = z0                                    on the last executed step (*last == step index),
//          = fp16(z0 + fp16(noise * fp16(sigma_next)))   otherwise (add_noise at the next sigma);
//   latents = fp16(fp16(fp16(1 - m) * proper) + fp16(m * latents)).
// The last step takes z0 itself, not add_noise with sigma 0: z0 + fp16(noise * 0) turns z0 = -0 into +0.
// mask: uint8 {0, 1} [Bm, hw]; latent image b uses mask b % Bm.  z0 / noise: fp16 NCHW, the latents' shape.
// ---------------------------------------------------------------------------------------------------------------
struct InpaintBlend {
  const unsigned char* mask;
  const __half* z0;
  const __half* noise;
  const int* last;
  long long hw;
  int Bm;
};

__device__ __forceinline__ __half inpaint_blend(const InpaintBlend& bl, long long idx, int img, long long e,
                                                bool last, float sig16_next, __half xh) {
  const float m = (float)bl.mask[(long long)(img % bl.Bm) * bl.hw + e % bl.hw];
  const float z = __half2float(bl.z0[idx]);
  const float proper =
      last ? z : __half2float(__float2half_rn(__fadd_rn(z, __half2float(__float2half_rn(
                                                              __fmul_rn(__half2float(bl.noise[idx]), sig16_next))))));
  const float keep = __half2float(__float2half_rn(__fmul_rn(__fsub_rn(1.f, m), proper)));
  const float gen = __half2float(__float2half_rn(__fmul_rn(m, __half2float(xh))));
  return __float2half_rn(__fadd_rn(keep, gen));
}

// ---------------------------------------------------------------------------------------------------------------
// CFG + Euler. Rounding points follow the reference's fp16 tensor arithmetic (custom_pipelines.py:348-350) and
// diffusers' EulerDiscreteScheduler.step (fp32 inside, result cast back to fp16).
// ---------------------------------------------------------------------------------------------------------------
template <bool BLEND>
__global__ void euler_cfg_kernel(const __half* __restrict__ noise, __half* __restrict__ latents,
                                 __half* __restrict__ model_in, const float* __restrict__ sigmas,
                                 const int* __restrict__ step, float guidance, long long per_image, int n_images,
                                 InpaintBlend bl) {
  pdl_launch_dependents();
  pdl_wait();
  const int i = *step;
  const float sigma = sigmas[i], sigma_next = sigmas[i + 1];
  const float den_next = sqrtf(sigma_next * sigma_next + 1.f);
  const long long total = per_image * n_images;
  bool last = false;
  float sig16_next = 0.f;
  if constexpr (BLEND) {
    last = i == *bl.last;
    sig16_next = __half2float(__float2half_rn(sigma_next));
  }
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const float u = __half2float(noise[idx]);
    const float c = __half2float(noise[total + idx]);
    const float d1 = __half2float(__float2half_rn(c - u));
    const float d2 = __half2float(__float2half_rn(guidance * d1));
    const float eps = __half2float(__float2half_rn(u + d2));
    const float x = __half2float(latents[idx]);
    // [3P] diffusers: `sample - sigma_hat * model_output` multiplies a 0-dim fp32 sigma with the fp16 model output,
    // so the product is an fp16 tensor (type promotion keeps the dimensioned tensor's dtype)
    const float x0 = x - __half2float(__float2half_rn(sigma * eps));
    const float deriv = (x - x0) / sigma;
    const float xn = x + deriv * (sigma_next - sigma);
    __half xh = __float2half_rn(xn);
    if constexpr (BLEND) {
      const int img = (int)(idx / per_image);
      xh = inpaint_blend(bl, idx, img, idx - (long long)img * per_image, last, sig16_next, xh);
    }
    latents[idx] = xh;
    const __half mi = __float2half_rn(__half2float(xh) / den_next);
    model_in[idx] = mi;
    model_in[total + idx] = mi;
  }
}
// General form of the step (custom_pipelines.py:346-357): classifier-free guidance on or off (:223,332,348) and the
// optional guidance rescale of :352-354 ([3P] diffusers rescale_noise_cfg: per-image unbiased std of the text branch
// and of the guided prediction over all non-batch elements, fp16 tensors -> fp16 rounding points).  ONE block per
// image: a first sweep forms the guided prediction and its statistics (double accumulators, fixed reduction order:
// deterministic), a second sweep -- the image is L1/L2 resident -- applies rescale + Euler.  n_images blocks of
// 1024 threads; a 4 x 128 x 128 latent is 64 elements per thread.
template <bool BLEND>
__global__ void __launch_bounds__(1024) euler_ex_kernel(const __half* __restrict__ noise, __half* __restrict__ latents,
                                                         __half* __restrict__ model_in,
                                                         const float* __restrict__ sigmas, const int* __restrict__ step,
                                                         float guidance, float rescale, long long per_image,
                                                         int n_images, int cfg, InpaintBlend bl) {
  pdl_launch_dependents();
  pdl_wait();
  const int img = blockIdx.x;
  const int i = *step;
  const float sigma = sigmas[i], sigma_next = sigmas[i + 1];
  const float den_next = sqrtf(sigma_next * sigma_next + 1.f);
  const long long total = per_image * n_images;
  const long long base = (long long)img * per_image;
  bool last = false;
  float sig16_next = 0.f;
  if constexpr (BLEND) {
    last = i == *bl.last;
    sig16_next = __half2float(__float2half_rn(sigma_next));
  }
  auto guided = [&](long long idx, float& c_out) -> float {
    if (!cfg) {
      c_out = __half2float(noise[idx]);
      return c_out;
    }
    const float u = __half2float(noise[idx]);
    const float c = __half2float(noise[total + idx]);
    c_out = c;
    const float d1 = __half2float(__float2half_rn(c - u));
    const float d2 = __half2float(__float2half_rn(guidance * d1));
    return __half2float(__float2half_rn(u + d2));
  };
  float factor = 1.f;   // fp16(std_text / std_cfg)
  if (cfg && rescale > 0.f) {
    double s_t = 0.0, q_t = 0.0, s_g = 0.0, q_g = 0.0;
    for (long long e = threadIdx.x; e < per_image; e += blockDim.x) {
      float c;
      const float g = guided(base + e, c);
      s_t += c;
      q_t += (double)c * c;
      s_g += g;
      q_g += (double)g * g;
    }
    __shared__ double red[4][32];
    __shared__ float s_factor;
    double v[4] = {s_t, q_t, s_g, q_g};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
      if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = v[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      double t[4] = {0, 0, 0, 0};
      const int nw = (blockDim.x + 31) >> 5;
      for (int k = 0; k < 4; ++k)
        for (int w = 0; w < nw; ++w) t[k] += red[k][w];
      const double n = (double)per_image;
      const double var_t = fmax((t[1] - t[0] * t[0] / n) / (n - 1.0), 0.0);
      const double var_g = fmax((t[3] - t[2] * t[2] / n) / (n - 1.0), 0.0);
      const float std_t = __half2float(__float2half_rn((float)sqrt(var_t)));   // torch.std of an fp16 tensor -> fp16
      const float std_g = __half2float(__float2half_rn((float)sqrt(var_g)));
      s_factor = __half2float(__float2half_rn(std_t / std_g));
    }
    __syncthreads();
    factor = s_factor;
  }
  for (long long e = threadIdx.x; e < per_image; e += blockDim.x) {
    const long long idx = base + e;
    float c;
    float eps = guided(idx, c);
    if (cfg && rescale > 0.f) {
      const float resc = __half2float(__float2half_rn(eps * factor));                  // noise_cfg * (std_text / std_cfg)
      const float a = __half2float(__float2half_rn(rescale * resc));
      const float b = __half2float(__float2half_rn((1.f - rescale) * eps));
      eps = __half2float(__float2half_rn(a + b));
    }
    const float x = __half2float(latents[idx]);
    const float x0 = x - __half2float(__float2half_rn(sigma * eps));
    const float deriv = (x - x0) / sigma;
    const float xn = x + deriv * (sigma_next - sigma);
    __half xh = __float2half_rn(xn);
    if constexpr (BLEND) xh = inpaint_blend(bl, idx, img, e, last, sig16_next, xh);
    latents[idx] = xh;
    const __half mi = __float2half_rn(__half2float(xh) / den_next);
    model_in[idx] = mi;
    if (cfg) model_in[total + idx] = mi;
  }
}

__global__ void step_inc_kernel(int* step) {
  pdl_launch_dependents();
  pdl_wait();
  *step += 1;
}

__global__ void scale_model_input_kernel(const __half* __restrict__ latents, __half* __restrict__ model_in,
                                         const float* __restrict__ sigmas, const int* __restrict__ step,
                                         long long total, int duplicate) {
  pdl_launch_dependents();
  pdl_wait();
  const float sigma = sigmas[*step];
  const float den = sqrtf(sigma * sigma + 1.f);
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const __half mi = __float2half_rn(__half2float(latents[idx]) / den);
    model_in[idx] = mi;
    if (duplicate) model_in[total + idx] = mi;   // CFG batch [uncond | cond] (custom_pipelines.py:332)
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Small generic attention (any head dims <= 128, few queries): one warp per (batch, head, query).
// HarmonyAttention's Cross_Attention (attention_processor.py:35-56): head_dim 40, value dim 64; scores are DIVIDED by
// `scale` = sqrt(head_dim) exactly like the reference (:45).
// ---------------------------------------------------------------------------------------------------------------
constexpr int SA_MAXK = 1024;
__global__ void attention_small_kernel(const __half* __restrict__ q, long long ldq, const __half* __restrict__ k,
                                       long long ldk, const __half* __restrict__ v, long long ldv,
                                       __half* __restrict__ out, long long ldo, int H, int Nq, int Nk, int dqk, int dv,
                                       float scale) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float s_p[];  // [warps][Nk]
  const int warp_in_block = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int gw = blockIdx.x * (blockDim.x >> 5) + warp_in_block;  // (b, h, iq)
  const int iq = gw % Nq;
  const int h = (gw / Nq) % H;
  const int b = gw / (Nq * H);
  float* p = s_p + warp_in_block * Nk;
  const __half* qr = q + ((long long)b * Nq + iq) * ldq + h * dqk;
  float mx = -INFINITY;
  for (int j = lane; j < Nk; j += 32) {
    const __half* kr = k + ((long long)b * Nk + j) * ldk + h * dqk;
    float acc = 0.f;
    for (int d = 0; d < dqk; ++d) acc += __half2float(qr[d]) * __half2float(kr[d]);
    // the reference rounds the fp16 matmul output before dividing by the scale (attention_processor.py:45)
    acc = __half2float(__float2half_rn(__half2float(__float2half_rn(acc)) / scale));
    p[j] = acc;
    mx = fmaxf(mx, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.f;
  for (int j = lane; j < Nk; j += 32) {
    const float e = __expf(p[j] - mx);
    p[j] = e;
    sum += e;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  __syncwarp();
  const float inv = 1.f / sum;
  for (int d = lane; d < dv; d += 32) {
    float acc = 0.f;
    for (int j = 0; j < Nk; ++j) {
      const float pj = __half2float(__float2half_rn(p[j] * inv));  // softmax output is an fp16 tensor
      acc += pj * __half2float(v[((long long)b * Nk + j) * ldv + h * dv + d]);
    }
    out[((long long)b * Nq + iq) * ldo + h * dv + d] = __float2half_rn(acc);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Generic SDPA for the CLIP towers (scope row f2: [3P] transformers CLIPAttention as the reference calls it through
// ip_adapter.py:81-84,163-164 (vision, head_dim 104 for ViT-bigG) and encode_prompt :292-319 (text, causal mask)):
// softmax(q k^T * scale [+ causal mask]) v with fp32 scores / softmax, one warp per (batch, head, query); keys are
// strided over the lanes with 16-byte loads, the PV sweep gives each lane dv/32 output channels.  head dims % 8 == 0.
// ---------------------------------------------------------------------------------------------------------------
__global__ void attention_generic_kernel(const __half* __restrict__ q, long long ldq, const __half* __restrict__ k,
                                         long long ldk, const __half* __restrict__ v, long long ldv,
                                         __half* __restrict__ out, long long ldo, int H, int Nq, int Nk, int dqk, int dv,
                                         float scale, int causal, long long total_warps) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float s_p[];  // [warps][Nk]
  const int warp_in_block = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const long long gw = (long long)blockIdx.x * (blockDim.x >> 5) + warp_in_block;  // (b, h, iq)
  if (gw >= total_warps) return;
  const int iq = (int)(gw % Nq);
  const int h = (int)((gw / Nq) % H);
  const int b = (int)(gw / ((long long)Nq * H));
  float* p = s_p + warp_in_block * Nk;
  const __half* qr = q + ((long long)b * Nq + iq) * ldq + h * dqk;
  const int nk_live = causal ? min(Nk, iq + 1 + (Nk - Nq)) : Nk;   // key j visible iff j <= iq (+ offset when Nk > Nq)
  float mx = -INFINITY;
  for (int j = lane; j < nk_live; j += 32) {
    const __half* kr = k + ((long long)b * Nk + j) * ldk + h * dqk;
    float acc = 0.f;
    for (int d = 0; d < dqk; d += 8) {
      float a[8], c[8];
      ld8(qr + d, a);
      ld8(kr + d, c);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc = fmaf(a[e], c[e], acc);
    }
    acc *= scale;
    p[j] = acc;
    mx = fmaxf(mx, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.f;
  for (int j = lane; j < nk_live; j += 32) {
    const float e = __expf(p[j] - mx);
    p[j] = e;
    sum += e;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  __syncwarp();
  const float inv = 1.f / sum;
  for (int d = lane; d < dv; d += 32) {
    float acc = 0.f;
    const __half* vc = v + (long long)b * Nk * ldv + h * dv + d;
    for (int j = 0; j < nk_live; ++j) acc = fmaf(p[j], __half2float(vc[(long long)j * ldv]), acc);
    out[((long long)b * Nq + iq) * ldo + h * dv + d] = __float2half_rn(acc * inv);
  }
}

// out[b, t, :] = tok_emb[ids[b, t], :] + pos_emb[t, :]   ([3P] CLIPTextEmbeddings; one 16-byte vector per thread)
__global__ void embed_tokens_kernel(const int* __restrict__ ids, const __half* __restrict__ tok, const __half* __restrict__ pos,
                                    __half* __restrict__ out, int rows, int T, int C8, int vocab) {
  pdl_launch_dependents();
  pdl_wait();
  const long long total = (long long)rows * C8;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / C8), c = (int)(i - (long long)r * C8);
    int id = ids[r];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    const uint4 a = reinterpret_cast<const uint4*>(tok)[(long long)id * C8 + c];
    const uint4 b = reinterpret_cast<const uint4*>(pos)[(long long)(r % T) * C8 + c];
    const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
    uint32_t o[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = unpack_half2(aw[e]), g = unpack_half2(bw[e]);
      o[e] = pack_half2(f.x + g.x, f.y + g.y);
    }
    reinterpret_cast<uint4*>(out)[i] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// CLIP-scorer front end (PNS judge): decoded image NCHW fp16 in [-1, 1] -> area-averaged S x S image -> [0, 1] ->
// (v - mean[c]) / std[c] -> patch rows [B * (S/P)^2, Kpad] with k = c*P*P + py*P + px (the layout of the flattened
// CLIP patch_embedding conv weight), zero padded to Kpad.  One thread per output pixel and channel.
__global__ void resize_patchify_kernel(const __half* __restrict__ img, __half* __restrict__ out, int B, int C, int Hin,
                                       int Win, int S, int P, int Kpad, float m0, float m1, float m2, float s0, float s1,
                                       float s2) {
  pdl_launch_dependents();
  pdl_wait();
  const int G = S / P;
  const long long total = (long long)B * G * G * Kpad;
  const float fy = (float)Hin / (float)S, fx = (float)Win / (float)S;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int kk = (int)(i % Kpad);
    const long long row = i / Kpad;
    if (kk >= C * P * P) {
      out[i] = __float2half_rn(0.f);
      continue;
    }
    const int c = kk / (P * P), py = (kk / P) % P, px = kk % P;
    const int gx = (int)(row % G), gy = (int)((row / G) % G), b = (int)(row / ((long long)G * G));
    const int oy = gy * P + py, ox = gx * P + px;
    const float y0 = oy * fy, y1 = (oy + 1) * fy, x0 = ox * fx, x1 = (ox + 1) * fx;
    const int iy0 = (int)floorf(y0), iy1 = min(Hin, (int)ceilf(y1)), ix0 = (int)floorf(x0), ix1 = min(Win, (int)ceilf(x1));
    const __half* src = img + ((long long)b * C + c) * Hin * Win;
    float acc = 0.f, wsum = 0.f;
    for (int y = iy0; y < iy1; ++y) {
      const float wy = fminf(y1, (float)(y + 1)) - fmaxf(y0, (float)y);
      for (int x = ix0; x < ix1; ++x) {
        const float wx = fminf(x1, (float)(x + 1)) - fmaxf(x0, (float)x);
        acc = fmaf(wy * wx, __half2float(src[(long long)y * Win + x]), acc);
        wsum += wy * wx;
      }
    }
    float vpx = fminf(fmaxf(acc / wsum * 0.5f + 0.5f, 0.f), 1.f);
    const float mean = c == 0 ? m0 : (c == 1 ? m1 : m2), sd = c == 0 ? s0 : (c == 1 ? s1 : s2);
    out[i] = __float2half_rn((vpx - mean) / sd);
  }
}

// out[i] = a[i] + b[i % period]  (16-byte vectors; period in elements, multiple of 8)
__global__ void add_bcast_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, uint4* __restrict__ out,
                                 long long nvec, long long period_vec) {
  pdl_launch_dependents();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    const uint4 x = a[i], y = b[i % period_vec];
    const uint32_t xw[4] = {x.x, x.y, x.z, x.w}, yw[4] = {y.x, y.y, y.z, y.w};
    uint32_t o[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = unpack_half2(xw[e]), g = unpack_half2(yw[e]);
      o[e] = pack_half2(f.x + g.x, f.y + g.y);
    }
    out[i] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// out[b, :] = mean over n of x[b, n, :]   (fp32 accumulation; one thread per 8 channels)
__global__ void mean_tokens_kernel(const __half* __restrict__ x, __half* __restrict__ out, int n, int D) {
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.y;
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (c >= D) return;
  float acc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] = 0.f;
  for (int i = 0; i < n; ++i) {
    float v[8];
    ld8(x + ((long long)b * n + i) * D + c, v);
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] += v[e];
  }
  uint4 o;
  const float inv = 1.f / (float)n;
  o.x = pack_half2(acc[0] * inv, acc[1] * inv);
  o.y = pack_half2(acc[2] * inv, acc[3] * inv);
  o.z = pack_half2(acc[4] * inv, acc[5] * inv);
  o.w = pack_half2(acc[6] * inv, acc[7] * inv);
  *reinterpret_cast<uint4*>(out + (long long)b * D + c) = o;
}

// Row softmax in place: x[r, :] <- softmax(x[r, :]) over `cols` fp16 values (fp32 statistics), one block per row, the row
// held in registers (cols <= 256 threads x 16 vectors x 8 = 32768).  Used by the single-head, head_dim 512 attention
// of the VAE decoder's mid block (scores = (q / sqrt(d)) k^T from the tensor-core GEMM).
constexpr int SMX_THREADS = 256;
constexpr int SMX_MAXV = 16;
__global__ void __launch_bounds__(SMX_THREADS) softmax_rows_kernel(__half* __restrict__ x, long long ld, int cols,
                                                                   int valid) {
  __shared__ float s_red[SMX_THREADS / 32];
  __shared__ float s_bcast;
  pdl_launch_dependents();
  pdl_wait();
  __half* row = x + (long long)blockIdx.x * ld;
  const int nv = cols >> 3;
  float v[SMX_MAXV][8];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < SMX_MAXV; ++i) {
    const int vi = threadIdx.x + i * SMX_THREADS;
    if (vi < nv) {
      ld8(row + vi * 8, v[i]);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        if (vi * 8 + e >= valid) v[i][e] = -INFINITY;   // padding columns (keys past the sequence end) get weight 0
        mx = fmaxf(mx, v[i][e]);
      }
    }
  }
  auto block_reduce = [&](float val, bool is_max) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float other = __shfl_xor_sync(0xffffffffu, val, o);
      val = is_max ? fmaxf(val, other) : val + other;
    }
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = val;
    __syncthreads();
    if (threadIdx.x == 0) {
      float r = s_red[0];
      for (int w = 1; w < SMX_THREADS / 32; ++w) r = is_max ? fmaxf(r, s_red[w]) : r + s_red[w];   // fixed order
      s_bcast = r;
    }
    __syncthreads();
    const float out = s_bcast;
    __syncthreads();
    return out;
  };
  mx = block_reduce(mx, true);
  const float ml2 = mx * 1.4426950408889634f;
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < SMX_MAXV; ++i) {
    const int vi = threadIdx.x + i * SMX_THREADS;
    if (vi < nv) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        v[i][e] = ex2_approx(fmaf(v[i][e], 1.4426950408889634f, -ml2));
        sum += v[i][e];
      }
    }
  }
  sum = block_reduce(sum, false);
  const float inv = 1.f / sum;
#pragma unroll
  for (int i = 0; i < SMX_MAXV; ++i) {
    const int vi = threadIdx.x + i * SMX_THREADS;
    if (vi < nv) {
      uint4 o;
      o.x = pack_half2(v[i][0] * inv, v[i][1] * inv);
      o.y = pack_half2(v[i][2] * inv, v[i][3] * inv);
      o.z = pack_half2(v[i][4] * inv, v[i][5] * inv);
      o.w = pack_half2(v[i][6] * inv, v[i][7] * inv);
      *reinterpret_cast<uint4*>(row + vi * 8) = o;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// The 4-channel ends of the UNet on the tensor-core GEMM:
//   conv_in : im2col of the NCHW latent -> A [B*H*W, 64] (k = ci*9 + ky*3 + kx, zero padded from 36 to 64 columns),
//             then ih_gemm_f16 with the OIHW weight flattened to [320, 36->64]
//   conv_out: ih_conv2d_f16 with Cout padded 4 -> 16, then this gather NHWC[.., 16] -> NCHW[B, 4, H, W]
// ---------------------------------------------------------------------------------------------------------------
__global__ void im2col3x3_nchw_kernel(const __half* __restrict__ x, __half* __restrict__ out, int B, int Cin, int H,
                                      int W, int Kpad) {
  pdl_launch_dependents();
  pdl_wait();
  const long long npix = (long long)B * H * W;
  const int kv = Kpad >> 3;  // 16-byte vectors per row
  const long long total = npix * kv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % kv);
    const long long pix = i / kv;
    const int xw = (int)(pix % W);
    const int yh = (int)((pix / W) % H);
    const int b = (int)(pix / ((long long)W * H));
    __align__(16) __half vals[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = v * 8 + e;
      __half hv = __float2half_rn(0.f);
      if (k < Cin * 9) {
        const int ci = k / 9, t = k - ci * 9;
        const int yy = yh + t / 3 - 1, xx = xw + t % 3 - 1;
        if (yy >= 0 && yy < H && xx >= 0 && xx < W) hv = x[(((long long)b * Cin + ci) * H + yy) * W + xx];
      }
      vals[e] = hv;
    }
    *reinterpret_cast<uint4*>(out + pix * Kpad + v * 8) = *reinterpret_cast<const uint4*>(vals);
  }
}

__global__ void nhwc_to_nchw_kernel(const __half* __restrict__ x, long long ldc, __half* __restrict__ out, int B,
                                    long long HW, int C) {
  pdl_launch_dependents();
  pdl_wait();
  const long long total = (long long)B * C * HW;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long p = i % HW;
    const int c = (int)((i / HW) % C);
    const int b = (int)(i / (HW * C));
    out[i] = x[((long long)b * HW + p) * ldc + c];
  }
}

// ---------------------------------------------------------------------------------------------------------------
// The two ends of the VAE encoder (img2img):
//   image front end: uint8 RGB NHWC (the PIL pixels) -> im2col rows [B*H*W, Kpad] of the normalised image for the
//                    encoder's conv_in GEMM.  Value = fp16(2 * (v / 255) - 1) with diffusers' fp32 rounding points
//                    (numpy `/ 255.0` in fp32, then `2 * x - 1` in fp32), zero padding 1, zero K padding.
//   sample + noise : z = fp16(sf * fp16(mean + exp(0.5 clamp(logvar, -30, 20)) * eps))  (DiagonalGaussianDistribution
//                    .sample in fp32, the cast to fp16, `scaling_factor * latents` in fp16), then
//                    fp16(z + fp16(noise * fp16(sigma)))  (EulerDiscreteScheduler.add_noise on fp16 tensors).
// ---------------------------------------------------------------------------------------------------------------
__global__ void image_im2col3x3_u8_kernel(const unsigned char* __restrict__ x, __half* __restrict__ out, int B, int H,
                                          int W, int Kpad) {
  pdl_launch_dependents();
  pdl_wait();
  const long long npix = (long long)B * H * W;
  const int kv = Kpad >> 3;
  const long long total = npix * kv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % kv);
    const long long pix = i / kv;
    const int xw = (int)(pix % W);
    const int yh = (int)((pix / W) % H);
    const int b = (int)(pix / ((long long)W * H));
    __align__(16) __half vals[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = v * 8 + e;
      __half hv = __float2half_rn(0.f);
      if (k < 27) {
        const int ci = k / 9, t = k - ci * 9;
        const int yy = yh + t / 3 - 1, xx = xw + t % 3 - 1;
        if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
          const float u = (float)x[(((long long)b * H + yy) * W + xx) * 3 + ci];
          hv = __float2half_rn(__fsub_rn(__fmul_rn(2.f, __fdiv_rn(u, 255.f)), 1.f));
        }
      }
      vals[e] = hv;
    }
    *reinterpret_cast<uint4*>(out + pix * Kpad + v * 8) = *reinterpret_cast<const uint4*>(vals);
  }
}

// INPAINT = true also writes z to z0_out (the blend's clean latents, fp16-exact) and, with pure_noise, sets
// out = fp16(noise * sigma) with sigma = init_noise_sigma unrounded (strength 1: `noise * init_noise_sigma`).
template <bool INPAINT>
__global__ void vae_sample_add_noise_kernel(const __half* __restrict__ moments, long long ldm, int Bm,
                                            const float* __restrict__ eps, int Be, const __half* __restrict__ noise,
                                            __half* __restrict__ out, int B, int C, long long HW, float sf, float sigma,
                                            __half* __restrict__ z0_out, int pure_noise) {
  pdl_launch_dependents();
  pdl_wait();
  const float sig16 = __half2float(__float2half_rn(sigma));
  const long long total = (long long)B * C * HW;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long p = i % HW;
    const int c = (int)((i / HW) % C);
    const int b = (int)(i / (HW * C));
    const __half* m = moments + ((long long)(b % Bm) * HW + p) * ldm;
    float z;
    if (eps) {
      const float lv = fminf(fmaxf(__half2float(m[C + c]), -30.f), 20.f);
      const float sd = expf(0.5f * lv);
      const float e = eps[((long long)(b % Be) * C + c) * HW + p];
      const float smp = __fadd_rn(__half2float(m[c]), __fmul_rn(sd, e));
      z = __half2float(__float2half_rn(__fmul_rn(__half2float(__float2half_rn(smp)), sf)));
    } else {
      z = __half2float(m[c]);                        // latents given as they are (4-channel image input)
    }
    if constexpr (INPAINT) {
      z0_out[i] = __float2half_rn(z);
      if (pure_noise) {
        out[i] = __float2half_rn(__fmul_rn(__half2float(noise[i]), sigma));
        continue;
      }
    }
    const float ns = __half2float(__float2half_rn(__fmul_rn(__half2float(noise[i]), sig16)));
    out[i] = __float2half_rn(__fadd_rn(z, ns));
  }
}

// Inpainting latent mask: uint8 grayscale [Bm, H, W] -> uint8 {0, 1} [Bm, H/8, W/8].  [3P] diffusers binarizes
// v / 255 at 0.5 (v >= 128 for uint8 pixels) and takes the latent mask with F.interpolate's default nearest mode, so
// latent (y, x) reads pixel (8y, 8x).
__global__ void latent_mask_u8_kernel(const unsigned char* __restrict__ mask, unsigned char* __restrict__ out, int Bm,
                                      int H, int W) {
  pdl_launch_dependents();
  pdl_wait();
  const int h = H / 8, w = W / 8;
  const long long total = (long long)Bm * h * w;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % w);
    const int y = (int)((i / w) % h);
    const int b = (int)(i / ((long long)w * h));
    out[i] = mask[((long long)b * H + 8 * y) * W + 8 * x] >= 128 ? 1 : 0;
  }
}

static int grid_for(long long total, int threads) {
  long long b = (total + threads - 1) / threads;
  const long long cap = (long long)num_sms() * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace ih

using namespace ih;

extern "C" int ih_linear_small_f16(const void* x, long long ldx, const void* w, const void* bias, const void* addend,
                                   long long ld_add, void* out, long long ldo, int M, int N, int K, int act_in,
                                   int act_out, float out_scale, void* stream) {
  IH_CHECK(x && w && out, IH_ERR_ARG, "ih_linear_small_f16: null pointer");
  IH_CHECK(M >= 1 && M <= 64, IH_ERR_SHAPE, "ih_linear_small_f16: M=%d must be in [1,64] (use ih_gemm_f16)", M);
  IH_CHECK(K % 8 == 0 && ldx % 8 == 0, IH_ERR_ALIGN, "ih_linear_small_f16: K and ldx must be multiples of 8");
  const int warps = 8;
  for (int m0 = 0; m0 < M; m0 += SL_MAXM) {  // row chunks of 8 (W is re-read from L2 for the later chunks)
    const int mc = (M - m0) < SL_MAXM ? (M - m0) : SL_MAXM;
    IH_CUDA(launch_kernel(linear_small_kernel, dim3((N + warps - 1) / warps), dim3(warps * 32), (size_t)(0), (cudaStream_t)stream, 
        (const __half*)x + m0 * ldx, ldx, (const __half*)w, (const __half*)bias,
        addend ? (const __half*)addend + m0 * ld_add : nullptr, ld_add, (__half*)out + m0 * ldo, ldo, mc, N, K,
        act_in, act_out, out_scale));
  }
  return 0;
}

extern "C" int ih_sinusoid_f16(const void* t_f32, const void* step_i32, void* out, long long ldo, int n, int dim,
                               void* stream) {
  IH_CHECK(t_f32 && out && dim % 2 == 0, IH_ERR_ARG, "ih_sinusoid_f16: bad arguments");
  const int total = n * (dim / 2);
  IH_CUDA(launch_kernel(sinusoid_kernel, dim3((total + 255) / 256), dim3(256), (size_t)(0), (cudaStream_t)stream, (const float*)t_f32, (const int*)step_i32,
                                                                         (__half*)out, ldo, n, dim));
  return 0;
}

extern "C" int ih_upsample2x_f16(const void* x, void* out, int B, int H, int W, int C, void* stream) {
  IH_CHECK(x && out && C % 8 == 0, IH_ERR_ARG, "ih_upsample2x_f16: bad arguments");
  const long long total = (long long)B * 4 * H * W * (C / 8);
  IH_CUDA(launch_kernel(upsample2x_kernel, dim3(grid_for(total, 256)), dim3(256), (size_t)(0), (cudaStream_t)stream, (const uint4*)x, (uint4*)out, B, H, W,
                                                                            C / 8));
  return 0;
}

extern "C" int ih_concat_f16(const void* x0, int C0, const void* x1, int C1, void* out, long long rows, void* stream) {
  IH_CHECK(x0 && x1 && out && C0 % 8 == 0 && C1 % 8 == 0, IH_ERR_ARG, "ih_concat_f16: bad arguments");
  const long long total = rows * ((C0 + C1) / 8);
  IH_CUDA(launch_kernel(concat_kernel, dim3(grid_for(total, 256)), dim3(256), (size_t)(0), (cudaStream_t)stream, (const uint4*)x0, C0 / 8, (const uint4*)x1,
                                                                        C1 / 8, (uint4*)out, rows));
  return 0;
}

extern "C" int ih_conv_in_f16(const void* x_nchw, const void* w, const void* bias, void* out, int B, int H, int W,
                              int Cin, int Cout, void* stream) {
  IH_CHECK(x_nchw && w && out, IH_ERR_ARG, "ih_conv_in_f16: null pointer");
  IH_CHECK(Cin <= 8 && Cout % 8 == 0 && Cin * 9 * Cout * 2 <= 48 * 1024, IH_ERR_SHAPE, "ih_conv_in_f16: bad shape");
  const long long total = (long long)B * H * W * (Cout / 8);
  IH_CUDA(launch_kernel(conv_in_kernel, dim3(grid_for(total, 256)), dim3(256), (size_t)(Cin * 9 * Cout * 2), (cudaStream_t)stream, 
      (const __half*)x_nchw, (const __half*)w, (const __half*)bias, (__half*)out, B, H, W, Cin, Cout));
  return 0;
}

extern "C" int ih_conv_out_f16(const void* x, const void* w, const void* bias, void* out_nchw, int B, int H, int W,
                               int Cin, int Cout, void* stream) {
  IH_CHECK(x && w && out_nchw, IH_ERR_ARG, "ih_conv_out_f16: null pointer");
  IH_CHECK(Cout <= CO_MAX && Cin % 8 == 0 && Cout * 9 * Cin * 2 <= 48 * 1024, IH_ERR_SHAPE,
           "ih_conv_out_f16: bad shape");
  const long long npix = (long long)B * H * W;
  long long blocks = (npix + 7) / 8;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  IH_CUDA(launch_kernel(conv_out_kernel, dim3((int)blocks), dim3(256), (size_t)(Cout * 9 * Cin * 2), (cudaStream_t)stream, 
      (const __half*)x, (const __half*)w, (const __half*)bias, (__half*)out_nchw, B, H, W, Cin, Cout));
  return 0;
}

extern "C" int ih_euler_cfg_step(const void* noise_pred, void* latents, void* model_in, const void* sigmas, void* step,
                                 float guidance, long long n_per_image, int n_images, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  IH_CHECK(noise_pred && latents && model_in && sigmas && step, IH_ERR_ARG, "ih_euler_cfg_step: null pointer");
  const long long total = n_per_image * n_images;
  IH_CUDA(launch_kernel(euler_cfg_kernel<false>, dim3(grid_for(total, 256)), dim3(256), (size_t)(0), stream, (const __half*)noise_pred, (__half*)latents,
                                                             (__half*)model_in, (const float*)sigmas,
                                                             (const int*)step, guidance, n_per_image, n_images,
                                                             InpaintBlend{}));
  IH_CUDA(launch_kernel(step_inc_kernel, dim3(1), dim3(1), (size_t)(0), stream, (int*)step));
  return 0;
}

extern "C" int ih_euler_step_ex(const void* noise_pred, void* latents, void* model_in, const void* sigmas, void* step,
                                float guidance, float guidance_rescale, long long n_per_image, int n_images,
                                int use_cfg, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  IH_CHECK(noise_pred && latents && model_in && sigmas && step, IH_ERR_ARG, "ih_euler_step_ex: null pointer");
  IH_CHECK(n_per_image > 1 && n_images > 0, IH_ERR_SHAPE, "ih_euler_step_ex: bad shape");
  IH_CHECK(guidance_rescale >= 0.f && guidance_rescale <= 1.f, IH_ERR_ARG, "ih_euler_step_ex: guidance_rescale outside [0, 1]");
  IH_CUDA(launch_kernel(euler_ex_kernel<false>, dim3(n_images), dim3(1024), (size_t)(0), stream, (const __half*)noise_pred,
                        (__half*)latents, (__half*)model_in, (const float*)sigmas, (const int*)step, guidance,
                        guidance_rescale, n_per_image, n_images, use_cfg ? 1 : 0, InpaintBlend{}));
  IH_CUDA(launch_kernel(step_inc_kernel, dim3(1), dim3(1), (size_t)(0), stream, (int*)step));
  return 0;
}

extern "C" int ih_euler_step_inpaint(const void* noise_pred, void* latents, void* model_in, const void* sigmas,
                                     void* step, float guidance, float guidance_rescale, long long n_per_image,
                                     int n_images, int use_cfg, const void* mask_u8, int Bm, long long hw,
                                     const void* z0, const void* noise, const void* last_step, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  IH_CHECK(noise_pred && latents && model_in && sigmas && step && mask_u8 && z0 && noise && last_step, IH_ERR_ARG,
           "ih_euler_step_inpaint: null pointer");
  IH_CHECK(n_per_image > 1 && n_images > 0 && hw > 0 && n_per_image % hw == 0 && Bm > 0 && n_images % Bm == 0,
           IH_ERR_SHAPE, "ih_euler_step_inpaint: bad shape (n_per_image %% hw == 0 and n_images %% Bm == 0 are required)");
  IH_CHECK(guidance_rescale >= 0.f && guidance_rescale <= 1.f, IH_ERR_ARG,
           "ih_euler_step_inpaint: guidance_rescale outside [0, 1]");
  const InpaintBlend bl{(const unsigned char*)mask_u8, (const __half*)z0, (const __half*)noise, (const int*)last_step,
                        hw, Bm};
  if (use_cfg && guidance_rescale == 0.f) {
    const long long total = n_per_image * n_images;
    IH_CUDA(launch_kernel(euler_cfg_kernel<true>, dim3(grid_for(total, 256)), dim3(256), (size_t)(0), stream,
                          (const __half*)noise_pred, (__half*)latents, (__half*)model_in, (const float*)sigmas,
                          (const int*)step, guidance, n_per_image, n_images, bl));
  } else {
    IH_CUDA(launch_kernel(euler_ex_kernel<true>, dim3(n_images), dim3(1024), (size_t)(0), stream,
                          (const __half*)noise_pred, (__half*)latents, (__half*)model_in, (const float*)sigmas,
                          (const int*)step, guidance, guidance_rescale, n_per_image, n_images, use_cfg ? 1 : 0, bl));
  }
  IH_CUDA(launch_kernel(step_inc_kernel, dim3(1), dim3(1), (size_t)(0), stream, (int*)step));
  return 0;
}

extern "C" int ih_scale_model_input(const void* latents, void* model_in, const void* sigmas, const void* step,
                                    long long total, void* stream) {
  return ih_scale_model_input_ex(latents, model_in, sigmas, step, total, 1, stream);
}

extern "C" int ih_scale_model_input_ex(const void* latents, void* model_in, const void* sigmas, const void* step,
                                       long long total, int duplicate, void* stream) {
  IH_CHECK(latents && model_in && sigmas && step, IH_ERR_ARG, "ih_scale_model_input: null pointer");
  IH_CUDA(launch_kernel(scale_model_input_kernel, dim3(grid_for(total, 256)), dim3(256), (size_t)(0), (cudaStream_t)stream, 
      (const __half*)latents, (__half*)model_in, (const float*)sigmas, (const int*)step, total, duplicate ? 1 : 0));
  return 0;
}

extern "C" int ih_attention_small_f16(const void* q, long long ldq, const void* k, long long ldk, const void* v,
                                      long long ldv, void* out, long long ldo, int B, int H, int Nq, int Nk, int dqk,
                                      int dv, float scale, void* stream) {
  IH_CHECK(q && k && v && out, IH_ERR_ARG, "ih_attention_small_f16: null pointer");
  IH_CHECK(Nk >= 1 && Nk <= SA_MAXK && dqk >= 1 && dqk <= 128 && dv >= 1 && dv <= 128 && Nq >= 1, IH_ERR_SHAPE,
           "ih_attention_small_f16: Nk<=%d, head dims <= 128 required", SA_MAXK);
  const int warps = 4;
  const long long total = (long long)B * H * Nq;
  IH_CHECK(total % warps == 0 || true, IH_ERR_SHAPE, "unreachable");
  const int blocks = (int)((total + warps - 1) / warps);
  // pad the grid so every warp index is valid: the kernel indexes (b,h,iq) from the global warp id
  IH_CHECK(total == (long long)blocks * warps, IH_ERR_SHAPE,
           "ih_attention_small_f16: B*H*Nq = %lld must be a multiple of %d", total, warps);
  IH_CUDA(launch_kernel(attention_small_kernel, dim3(blocks), dim3(warps * 32), (size_t)(warps * Nk * sizeof(float)), (cudaStream_t)stream, 
      (const __half*)q, ldq, (const __half*)k, ldk, (const __half*)v, ldv, (__half*)out, ldo, H, Nq, Nk, dqk, dv,
      scale));
  return 0;
}

extern "C" int ih_attention_generic_f16(const void* q, long long ldq, const void* k, long long ldk, const void* v,
                                        long long ldv, void* out, long long ldo, int B, int H, int Nq, int Nk, int dqk,
                                        int dv, float scale, int causal, void* stream) {
  IH_CHECK(q && k && v && out, IH_ERR_ARG, "ih_attention_generic_f16: null pointer");
  IH_CHECK(Nk >= 1 && Nk <= 4096 && Nq >= 1 && dqk >= 8 && dqk <= 256 && dv >= 1 && dv <= 256 && dqk % 8 == 0 &&
               ldq % 8 == 0 && ldk % 8 == 0, IH_ERR_SHAPE,
           "ih_attention_generic_f16: Nk <= 4096, head dims <= 256, dqk / ldq / ldk multiples of 8 required");
  IH_CHECK(!causal || Nk >= Nq, IH_ERR_SHAPE, "ih_attention_generic_f16: causal needs Nk >= Nq");
  const int warps = 4;
  const long long total = (long long)B * H * Nq;
  const int blocks = (int)((total + warps - 1) / warps);
  const size_t smem = (size_t)warps * Nk * sizeof(float);
  static bool configured = false;
  if (!configured) {
    IH_CUDA(cudaFuncSetAttribute(attention_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * 4096 * 4));
    configured = true;
  }
  IH_CUDA(launch_kernel(attention_generic_kernel, dim3(blocks), dim3(warps * 32), smem, (cudaStream_t)stream,
                        (const __half*)q, ldq, (const __half*)k, ldk, (const __half*)v, ldv, (__half*)out, ldo, H, Nq, Nk,
                        dqk, dv, scale, causal ? 1 : 0, total));
  return 0;
}

extern "C" int ih_embed_tokens_f16(const void* ids_i32, const void* tok_emb, const void* pos_emb, void* out, int rows,
                                   int T, int C, int vocab, void* stream) {
  IH_CHECK(ids_i32 && tok_emb && pos_emb && out, IH_ERR_ARG, "ih_embed_tokens_f16: null pointer");
  IH_CHECK(rows > 0 && T > 0 && C % 8 == 0 && vocab > 0, IH_ERR_SHAPE, "ih_embed_tokens_f16: bad shape");
  const long long total = (long long)rows * (C / 8);
  IH_CUDA(launch_kernel(embed_tokens_kernel, dim3(grid_for(total, 256)), dim3(256), (size_t)0, (cudaStream_t)stream,
                        (const int*)ids_i32, (const __half*)tok_emb, (const __half*)pos_emb, (__half*)out, rows, T, C / 8,
                        vocab));
  return 0;
}

extern "C" int ih_resize_patchify_f16(const void* img_nchw, void* out, int B, int C, int Hin, int Win, int S, int P,
                                      int Kpad, const float* mean3, const float* std3, void* stream) {
  IH_CHECK(img_nchw && out && mean3 && std3, IH_ERR_ARG, "ih_resize_patchify_f16: null pointer");
  IH_CHECK(C == 3 && S % P == 0 && Kpad % 8 == 0 && Kpad >= C * P * P && Hin > 0 && Win > 0, IH_ERR_SHAPE,
           "ih_resize_patchify_f16: 3 channels, S %% P == 0, Kpad >= 3*P*P (multiple of 8) required");
  const long long total = (long long)B * (S / P) * (S / P) * Kpad;
  IH_CUDA(launch_kernel(resize_patchify_kernel, dim3(grid_for(total, 256)), dim3(256), (size_t)0, (cudaStream_t)stream,
                        (const __half*)img_nchw, (__half*)out, B, C, Hin, Win, S, P, Kpad, mean3[0], mean3[1], mean3[2],
                        std3[0], std3[1], std3[2]));
  return 0;
}

extern "C" int ih_add_bcast_f16(const void* a, const void* b, void* out, long long n, long long period, void* stream) {
  IH_CHECK(a && b && out && n % 8 == 0 && period % 8 == 0 && period > 0, IH_ERR_ARG, "ih_add_bcast_f16: bad arguments");
  IH_CUDA(launch_kernel(add_bcast_kernel, dim3(grid_for(n / 8, 256)), dim3(256), (size_t)0, (cudaStream_t)stream,
                        (const uint4*)a, (const uint4*)b, (uint4*)out, n / 8, period / 8));
  return 0;
}

extern "C" int ih_mean_tokens_f16(const void* x, void* out, int B, int n, int D, void* stream) {
  IH_CHECK(x && out && D % 8 == 0 && n > 0, IH_ERR_ARG, "ih_mean_tokens_f16: bad arguments");
  IH_CUDA(launch_kernel(mean_tokens_kernel, dim3((D / 8 + 127) / 128, B), dim3(128), (size_t)0, (cudaStream_t)stream,
                        (const __half*)x, (__half*)out, n, D));
  return 0;
}

extern "C" int ih_softmax_rows_f16(void* x, long long ld, long long rows, int cols, void* stream) {
  IH_CHECK(x && rows > 0 && cols > 0, IH_ERR_ARG, "ih_softmax_rows_f16: bad arguments");
  IH_CHECK(cols % 8 == 0 && ld % 8 == 0 && cols <= SMX_THREADS * SMX_MAXV * 8, IH_ERR_SHAPE,
           "ih_softmax_rows_f16: cols must be a multiple of 8 and <= %d", SMX_THREADS * SMX_MAXV * 8);
  IH_CHECK(rows <= 0x7fffffffLL, IH_ERR_SHAPE, "ih_softmax_rows_f16: too many rows");
  IH_CUDA(launch_kernel(softmax_rows_kernel, dim3((unsigned)rows), dim3(SMX_THREADS), (size_t)0, (cudaStream_t)stream,
                        (__half*)x, ld, cols, cols));
  return 0;
}

extern "C" int ih_softmax_rows_masked_f16(void* x, long long ld, long long rows, int cols, int valid_cols, void* stream) {
  IH_CHECK(x && rows > 0 && cols > 0 && valid_cols > 0 && valid_cols <= cols, IH_ERR_ARG,
           "ih_softmax_rows_masked_f16: bad arguments");
  IH_CHECK(cols % 8 == 0 && ld % 8 == 0 && cols <= SMX_THREADS * SMX_MAXV * 8, IH_ERR_SHAPE,
           "ih_softmax_rows_masked_f16: cols must be a multiple of 8 and <= %d", SMX_THREADS * SMX_MAXV * 8);
  IH_CHECK(rows <= 0x7fffffffLL, IH_ERR_SHAPE, "ih_softmax_rows_masked_f16: too many rows");
  IH_CUDA(launch_kernel(softmax_rows_kernel, dim3((unsigned)rows), dim3(SMX_THREADS), (size_t)0, (cudaStream_t)stream,
                        (__half*)x, ld, cols, valid_cols));
  return 0;
}

extern "C" int ih_im2col3x3_nchw_f16(const void* x_nchw, void* out, int B, int Cin, int H, int W, int Kpad,
                                     void* stream) {
  IH_CHECK(x_nchw && out && Kpad % 8 == 0 && Kpad >= Cin * 9, IH_ERR_ARG, "ih_im2col3x3_nchw_f16: bad arguments");
  const long long total = (long long)B * H * W * (Kpad / 8);
  IH_CUDA(launch_kernel(im2col3x3_nchw_kernel, dim3(grid_for(total, 256)), dim3(256), (size_t)0, (cudaStream_t)stream,
                        (const __half*)x_nchw, (__half*)out, B, Cin, H, W, Kpad));
  return 0;
}

extern "C" int ih_nhwc_to_nchw_f16(const void* x, long long ldc, void* out, int B, long long HW, int C, void* stream) {
  IH_CHECK(x && out && C >= 1, IH_ERR_ARG, "ih_nhwc_to_nchw_f16: bad arguments");
  const long long total = (long long)B * C * HW;
  IH_CUDA(launch_kernel(nhwc_to_nchw_kernel, dim3(grid_for(total, 256)), dim3(256), (size_t)0, (cudaStream_t)stream,
                        (const __half*)x, ldc, (__half*)out, B, HW, C));
  return 0;
}

extern "C" int ih_image_im2col3x3_u8(const void* rgb_u8, void* out, int B, int H, int W, int Kpad, void* stream) {
  IH_CHECK(rgb_u8 && out, IH_ERR_ARG, "ih_image_im2col3x3_u8: null pointer");
  IH_CHECK(B > 0 && H > 0 && W > 0 && Kpad % 8 == 0 && Kpad >= 27, IH_ERR_SHAPE, "ih_image_im2col3x3_u8: bad shape");
  const long long total = (long long)B * H * W * (Kpad / 8);
  IH_CUDA(launch_kernel(image_im2col3x3_u8_kernel, dim3(grid_for(total, 256)), dim3(256), (size_t)0, (cudaStream_t)stream,
                        (const unsigned char*)rgb_u8, (__half*)out, B, H, W, Kpad));
  return 0;
}

extern "C" int ih_vae_sample_add_noise_f16(const void* moments, long long ldm, int Bm, const void* eps_f32, int Be,
                                           const void* noise, void* out_nchw, int B, int C, int h, int w,
                                           float scaling_factor, float sigma, void* stream) {
  IH_CHECK(moments && noise && out_nchw, IH_ERR_ARG, "ih_vae_sample_add_noise_f16: null pointer");
  IH_CHECK(B > 0 && C > 0 && h > 0 && w > 0 && Bm > 0 && B % Bm == 0 && ldm >= (eps_f32 ? 2 * C : C), IH_ERR_SHAPE,
           "ih_vae_sample_add_noise_f16: bad shape (B %% Bm == 0 and ldm >= 2C with eps, >= C without are required)");
  IH_CHECK(!eps_f32 || (Be > 0 && B % Be == 0), IH_ERR_SHAPE, "ih_vae_sample_add_noise_f16: B %% Be != 0");
  const long long HW = (long long)h * w;
  const long long total = (long long)B * C * HW;
  IH_CUDA(launch_kernel(vae_sample_add_noise_kernel<false>, dim3(grid_for(total, 256)), dim3(256), (size_t)0,
                        (cudaStream_t)stream, (const __half*)moments, ldm, Bm, (const float*)eps_f32, Be,
                        (const __half*)noise, (__half*)out_nchw, B, C, HW, scaling_factor, sigma, (__half*)nullptr, 0));
  return 0;
}

extern "C" int ih_vae_sample_inpaint_f16(const void* moments, long long ldm, int Bm, const void* eps_f32, int Be,
                                         const void* noise, void* latents_nchw, void* z0_nchw, int B, int C, int h,
                                         int w, float scaling_factor, float sigma, int pure_noise, void* stream) {
  IH_CHECK(moments && noise && latents_nchw && z0_nchw, IH_ERR_ARG, "ih_vae_sample_inpaint_f16: null pointer");
  IH_CHECK(B > 0 && C > 0 && h > 0 && w > 0 && Bm > 0 && B % Bm == 0 && ldm >= (eps_f32 ? 2 * C : C), IH_ERR_SHAPE,
           "ih_vae_sample_inpaint_f16: bad shape (B %% Bm == 0 and ldm >= 2C with eps, >= C without are required)");
  IH_CHECK(!eps_f32 || (Be > 0 && B % Be == 0), IH_ERR_SHAPE, "ih_vae_sample_inpaint_f16: B %% Be != 0");
  const long long HW = (long long)h * w;
  const long long total = (long long)B * C * HW;
  IH_CUDA(launch_kernel(vae_sample_add_noise_kernel<true>, dim3(grid_for(total, 256)), dim3(256), (size_t)0,
                        (cudaStream_t)stream, (const __half*)moments, ldm, Bm, (const float*)eps_f32, Be,
                        (const __half*)noise, (__half*)latents_nchw, B, C, HW, scaling_factor, sigma, (__half*)z0_nchw,
                        pure_noise ? 1 : 0));
  return 0;
}

extern "C" int ih_latent_mask_u8(const void* mask_u8, void* out_u8, int Bm, int H, int W, void* stream) {
  IH_CHECK(mask_u8 && out_u8, IH_ERR_ARG, "ih_latent_mask_u8: null pointer");
  IH_CHECK(Bm > 0 && H > 0 && W > 0 && H % 8 == 0 && W % 8 == 0, IH_ERR_SHAPE,
           "ih_latent_mask_u8: bad shape (H and W must be positive multiples of 8)");
  const long long total = (long long)Bm * (H / 8) * (W / 8);
  IH_CUDA(launch_kernel(latent_mask_u8_kernel, dim3(grid_for(total, 256)), dim3(256), (size_t)0, (cudaStream_t)stream,
                        (const unsigned char*)mask_u8, (unsigned char*)out_u8, Bm, H, W));
  return 0;
}
