// kernels_elem.cu -- elementwise / layout kernels and the fused per-step scheduler kernels.
//
// Scheduler kernels restate, op for op and with round-to-nearest intrinsics (no FMA contraction), the reference's
// per-step tensor arithmetic so that they are bit-exact against the reference CPU path:
//   ddim_posterior_sample   DDIMSampler.sample_xt_next          ddim.py:582-601
//   ddim_compute_eps        CFG combine + compute_eps tail      ddim.py:555-559, 575-579
//   ddim_step_with_eps      CFG combine + p_sample_ddim_with_eps tail   ddim.py:613-617, 634-645
//   pixel_*                 sample_xt_next / compute_eps / denoising_step_with_eps   ddpm_ddim_wrapper.py:114-307
//   pixel_lock_step         the three above for a source and a target chain in one launch (two-model lock-step cycle)
//   vae_posterior           DiagonalGaussianDistribution.sample * scale_factor      distributions.py:24-37, ddpm.py:536-543
// Each is one launch instead of the reference's ~8-10 elementwise launches per step (SURVEY.md 2.2).
#include "common.cuh"

namespace cdx {
namespace {

#define MUL(a, b) __fmul_rn((a), (b))
#define ADD(a, b) __fadd_rn((a), (b))
#define SUB(a, b) __fsub_rn((a), (b))
#define DIV(a, b) __fdiv_rn((a), (b))

inline int grid_for(size_t n, int num_sms) {
  size_t b = (n + 255) / 256;
  size_t cap = (size_t)num_sms * 16;
  return (int)(b < cap ? (b ? b : 1) : cap);
}
#define GRID_STRIDE(i, n) for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (n); i += (size_t)gridDim.x * blockDim.x)

__global__ void affine_kernel(const float* __restrict__ x, float a, float b, float* __restrict__ y, size_t n) {
  GRID_STRIDE(i, n) y[i] = ADD(MUL(a, x[i]), b);
}
__global__ void shift_scale_kernel(const float* __restrict__ x, float b, float a, float* __restrict__ y, size_t n) {
  GRID_STRIDE(i, n) y[i] = MUL(ADD(x[i], b), a);
}
__global__ void q_sample_kernel(const float* __restrict__ x0, const float* __restrict__ nz, float sa, float s1, float* __restrict__ y, size_t n) {
  GRID_STRIDE(i, n) y[i] = ADD(MUL(sa, x0[i]), MUL(s1, nz[i]));
}
__global__ void silu_kernel(const float* __restrict__ x, float* __restrict__ y, size_t n) {
  GRID_STRIDE(i, n) { const float v = x[i]; y[i] = v / (1.f + expf(-v)); }
}
__global__ void add_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ y, size_t n) {
  GRID_STRIDE(i, n) y[i] = a[i] + b[i];
}
__global__ void copy_kernel(const float* __restrict__ a, float* __restrict__ y, size_t n) {
  GRID_STRIDE(i, n) y[i] = a[i];
}
// x [M,2C] -> y [M,C] = x[:, :C] * gelu_erf(x[:, C:])   (attention.py:42-44)
__global__ void geglu_kernel(const float* __restrict__ x, float* __restrict__ y, size_t M, int C, int interleaved) {
  const size_t n = M * (size_t)C;
  GRID_STRIDE(i, n) {
    const size_t m = i / C;
    const int c = (int)(i - m * C);
    const int cv = interleaved ? ((c >> 5) << 6) + (c & 31) : c;      // [32 value | 32 gate] blocks (see Param::geglu)
    const int cg = interleaved ? cv + 32 : C + c;
    const float v = x[m * 2 * C + cv];
    const float g = x[m * 2 * C + cg];
    y[i] = v * (0.5f * g * (1.f + erff(g * 0.70710678118654752440f)));
  }
}
// rows [0, rows/2) are value rows, [rows/2, rows) gate rows -> blocks of 32 value rows followed by their 32 gate rows
__global__ void interleave_geglu_rows_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int rowlen) {
  const size_t n = (size_t)rows * rowlen;
  const int half = rows / 2;
  GRID_STRIDE(i, n) {
    const int r = (int)(i / rowlen);
    const int c = (int)(i - (size_t)r * rowlen);
    const int j = r < half ? r : r - half;
    const int dr = ((j >> 5) << 6) + (j & 31) + (r < half ? 0 : 32);
    dst[(size_t)dr * rowlen + c] = src[i];
  }
}
__global__ void avgpool2_kernel(const float* __restrict__ x, float* __restrict__ y, int B, int H, int W, int C) {
  const int Ho = H / 2, Wo = W / 2;
  const size_t n = (size_t)B * Ho * Wo * C;
  GRID_STRIDE(i, n) {
    const int c = (int)(i % C);
    size_t r = i / C;
    const int ox = (int)(r % Wo); r /= Wo;
    const int oy = (int)(r % Ho);
    const int b = (int)(r / Ho);
    const float* p = x + (((size_t)b * H + 2 * oy) * W + 2 * ox) * C + c;
    // ATen avg_pool2d sums the window then divides
    y[i] = (p[0] + p[C] + p[(size_t)W * C] + p[(size_t)W * C + C]) * 0.25f;
  }
}
__global__ void upsample2_kernel(const float* __restrict__ x, float* __restrict__ y, int B, int H, int W, int C) {
  const int Ho = H * 2, Wo = W * 2;
  const size_t n = (size_t)B * Ho * Wo * C;
  GRID_STRIDE(i, n) {
    const int c = (int)(i % C);
    size_t r = i / C;
    const int ox = (int)(r % Wo); r /= Wo;
    const int oy = (int)(r % Ho);
    const int b = (int)(r / Ho);
    y[i] = x[(((size_t)b * H + (oy >> 1)) * W + (ox >> 1)) * C + c];
  }
}
// tiled transposes between [B,C,HW] and [B,HW,C]
__global__ void transpose_kernel(const float* __restrict__ x, float* __restrict__ y, int R, int Cc) {
  // x: [b][R][Cc] -> y: [b][Cc][R]
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const float* xb = x + (size_t)b * R * Cc;
  float* yb = y + (size_t)b * R * Cc;
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int r = r0 + j, c = c0 + threadIdx.x;
    if (r < R && c < Cc) tile[j][threadIdx.x] = xb[(size_t)r * Cc + c];
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int c = c0 + j, r = r0 + threadIdx.x;
    if (r < R && c < Cc) yb[(size_t)c * R + r] = tile[threadIdx.x][j];
  }
}
// [cos | sin] (util.py:152-172, nn.py:103-122) or, sin_first, [sin | cos] (ddpm/diffusion.py:6-25)
__global__ void temb_kernel(const float* __restrict__ t, const float* __restrict__ freqs, float* __restrict__ emb, int B, int half, int sin_first) {
  const int n = B * half;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int b = i / half, j = i - b * half;
    const float a = MUL(t[b], freqs[j]);
    emb[(size_t)b * 2 * half + (sin_first ? half : 0) + j] = cosf(a);
    emb[(size_t)b * 2 * half + (sin_first ? 0 : half) + j] = sinf(a);
  }
}
// OIHW (3x3) -> O,kh,kw,I
// OIHW -> O,kh,kw,Ip with the input channels zero-padded from I to Ip (Ip == I: plain repack)
__global__ void repack_conv_kernel(const float* __restrict__ w, float* __restrict__ o, int O, int I, int Ip) {
  const size_t n = (size_t)O * Ip * 9;
  GRID_STRIDE(idx, n) {
    const int i = (int)(idx % Ip);
    size_t r = idx / Ip;
    const int tap = (int)(r % 9);
    const int oc = (int)(r / 9);
    o[idx] = i < I ? w[((size_t)oc * I + i) * 9 + tap] : 0.f;
  }
}
// CLIPTextEmbeddings: out[b, l, :] = token_embedding[ids[b, l]] + position_embedding[l]
__global__ void embed_tokens_kernel(const int* __restrict__ ids, const float* __restrict__ tok, const float* __restrict__ pos,
                                    float* __restrict__ out, int B, int L, int W, int vocab) {
  const size_t n = (size_t)B * L * W;
  GRID_STRIDE(idx, n) {
    const int c = (int)(idx % W);
    const size_t bl = idx / W;
    const int l = (int)(bl % L);
    int id = ids[bl];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    out[idx] = tok[(size_t)id * W + c] + pos[(size_t)l * W + c];
  }
}
// quick-GELU (HF activations.QuickGELUActivation): x * sigmoid(1.702 x)
__global__ void quick_gelu_kernel(const float* __restrict__ x, float* __restrict__ y, size_t n) {
  GRID_STRIDE(i, n) {
    const float v = x[i];
    y[i] = v * (1.f / (1.f + expf(-1.702f * v)));
  }
}
// exact (erf) GELU, nn.GELU() default
__global__ void gelu_kernel(const float* __restrict__ x, float* __restrict__ y, size_t n) {
  GRID_STRIDE(i, n) {
    const float v = x[i];
    y[i] = 0.5f * v * (1.f + erff(v * 0.70710678118654752440f));
  }
}
// x [rows][C] -> y [rows][Cp], zero fill
__global__ void pad_channels_kernel(const float* __restrict__ x, float* __restrict__ y, size_t rows, int C, int Cp) {
  const size_t n = rows * (size_t)Cp;
  GRID_STRIDE(idx, n) {
    const int c = (int)(idx % Cp);
    const size_t r = idx / Cp;
    y[idx] = c < C ? x[r * C + c] : 0.f;
  }
}

__global__ void vae_posterior_kernel(const float* __restrict__ mom, const float* __restrict__ nz, float sf, float* __restrict__ out,
                                     int B, int C, int hw) {
  const size_t n = (size_t)B * C * hw;
  GRID_STRIDE(i, n) {
    const size_t b = i / ((size_t)C * hw);
    const size_t r = i - b * (size_t)C * hw;
    const float mean = mom[b * 2 * C * hw + r];
    float z = mean;
    if (nz) {
      float lv = mom[b * 2 * C * hw + (size_t)C * hw + r];
      lv = fminf(fmaxf(lv, -30.0f), 20.0f);
      const float sd = expf(MUL(0.5f, lv));
      z = ADD(mean, MUL(sd, nz[i]));
    }
    out[i] = MUL(sf, z);
  }
}

__device__ __forceinline__ float cfg_combine(const float* e_c, const float* e_uc, float scale, size_t i) {
  const float ec = e_c[i];
  if (e_uc == nullptr) return ec;
  const float eu = e_uc[i];
  return ADD(eu, MUL(scale, SUB(ec, eu)));      // e_t_uncond + s * (e_t - e_t_uncond), ddim.py:559
}

// per-sample scale (ensemble batching): members whose scale is 1 or 0 take the reference's single-forward value bit for bit
__device__ __forceinline__ float cfg_combine_v(const float* e_c, const float* e_uc, float scale, size_t i) {
  const float ec = e_c[i];
  if (e_uc == nullptr || scale == 1.0f) return ec;
  const float eu = e_uc[i];
  if (scale == 0.0f) return eu;
  return ADD(eu, MUL(scale, SUB(ec, eu)));
}

__global__ void ddim_posterior_kernel(const float* __restrict__ x0, const float* __restrict__ xt, const float* __restrict__ nz,
                                      cdx_ddim_coef c, float* __restrict__ out, size_t n) {
  GRID_STRIDE(i, n) {
    const float e_t = DIV(SUB(xt[i], MUL(c.sqrt_at, x0[i])), c.sqrt_1m_at);       // ddim.py:597
    const float dir = MUL(c.dir_coef, e_t);                                       // :598
    const float noise = MUL(c.sigma, nz[i]);                                      // :599
    out[i] = ADD(ADD(MUL(c.sqrt_aprev, x0[i]), dir), noise);                      // :600
  }
}
__global__ void ddim_compute_eps_kernel(const float* __restrict__ xt, const float* __restrict__ xn, const float* __restrict__ e_c,
                                        const float* __restrict__ e_uc, float scale, cdx_ddim_coef c, float* __restrict__ out, size_t n) {
  GRID_STRIDE(i, n) {
    const float e_t = cfg_combine(e_c, e_uc, scale, i);
    const float pred_x0 = DIV(SUB(xt[i], MUL(c.sqrt_1m_at_tab, e_t)), c.sqrt_at);          // ddim.py:576
    const float dir = MUL(c.dir_coef, e_t);                                                // :578
    out[i] = DIV(DIV(SUB(SUB(xn[i], MUL(c.sqrt_aprev, pred_x0)), dir), c.sigma), 1.0f);    // :579 (temperature 1)
  }
}
__global__ void ddim_step_kernel(const float* __restrict__ x, const float* __restrict__ e_c, const float* __restrict__ e_uc, float scale,
                                 const float* __restrict__ eps, cdx_ddim_coef c, float* __restrict__ out, size_t n) {
  GRID_STRIDE(i, n) {
    const float e_t = cfg_combine(e_c, e_uc, scale, i);
    const float pred_x0 = DIV(SUB(x[i], MUL(c.sqrt_1m_at_tab, e_t)), c.sqrt_at);           // ddim.py:634
    const float dir = MUL(c.dir_coef, e_t);                                                // :638
    const float noise = MUL(MUL(c.sigma, eps[i]), 1.0f);                                   // :642
    out[i] = ADD(ADD(MUL(c.sqrt_aprev, pred_x0), dir), noise);                             // :645
  }
}

__device__ __forceinline__ float ddim_posterior_f(float x0, float xt, float nz, const cdx_ddim_coef& c) {
  const float e_t = DIV(SUB(xt, MUL(c.sqrt_at, x0)), c.sqrt_1m_at);       // ddim.py:597
  const float dir = MUL(c.dir_coef, e_t);                                 // :598
  const float noise = MUL(c.sigma, nz);                                   // :599
  return ADD(ADD(MUL(c.sqrt_aprev, x0), dir), noise);                     // :600
}

__global__ void latent_step_kernel(const LatentStep a) {
  const size_t seg = a.n;
  GRID_STRIDE(i, a.n) {
    const size_t b = i / a.chw, r = i - b * a.chw;
    float eps = 0.f;
    if (a.enc) {
      const float e_t = a.s_scale_v ? cfg_combine_v(a.es_c, a.es_uc, a.s_scale_v[b], i) : cfg_combine(a.es_c, a.es_uc, a.s_scale, i);
      const float xt = a.xt[i], xn = a.xn[i];
      const float pred_x0 = DIV(SUB(xt, MUL(a.cs.sqrt_1m_at_tab, e_t)), a.cs.sqrt_at);          // ddim.py:576
      const float dir = MUL(a.cs.dir_coef, e_t);                                                // :578
      eps = DIV(DIV(SUB(SUB(xn, MUL(a.cs.sqrt_aprev, pred_x0)), dir), a.cs.sigma), 1.0f);       // :579 (temperature 1)
      if (a.z_out) a.z_out[b * a.z_stride + r] = eps;
      if (a.next == 1) a.xn2[i] = ddim_posterior_f(a.x0[i], xn, a.noise_next[i], a.cnext);
      else if (a.next == 2) a.xn2[i] = a.x0[i];                                                 // ddim.py:583-584
      for (int sg = 0; sg < a.nseg_src; ++sg) a.xin[sg * seg + i] = xn;
    } else if (a.dec) {
      eps = a.eps_in[b * a.eps_stride + r];
    }
    if (a.dec) {
      const float e_t = a.t_scale_v ? cfg_combine_v(a.et_c, a.et_uc, a.t_scale_v[b], i) : cfg_combine(a.et_c, a.et_uc, a.t_scale, i);
      const float y = a.yt[i];
      const float pred_x0 = DIV(SUB(y, MUL(a.ct.sqrt_1m_at_tab, e_t)), a.ct.sqrt_at);           // ddim.py:634
      const float dir = MUL(a.ct.dir_coef, e_t);                                                // :638
      const float noise = MUL(MUL(a.ct.sigma, eps), 1.0f);                                      // :642
      const float yn = ADD(ADD(MUL(a.ct.sqrt_aprev, pred_x0), dir), noise);                     // :645
      a.y_out[i] = yn;
      for (int sg = 0; sg < a.nseg_tgt; ++sg) a.xin[(a.nseg_src + sg) * seg + i] = yn;
    }
  }
}

__global__ void latent_init_kernel(const LatentInit a) {
  const size_t seg = a.n;
  GRID_STRIDE(i, a.n) {
    const size_t b = i / a.chw, r = i - b * a.chw;
    const float x0 = a.x0[i];
    const float xT = ADD(MUL(a.sa, x0), MUL(a.s1, a.noise0[i]));                                // ddim.py:477-479
    if (a.z_out) a.z_out[b * a.z_stride + r] = xT;
    a.xt[i] = xT;
    if (a.yt) a.yt[i] = xT;
    if (a.next == 1) a.xn[i] = ddim_posterior_f(x0, xT, a.noise_next[i], a.cnext);
    else if (a.next == 2) a.xn[i] = x0;
    for (int sg = 0; sg < a.nseg_src + a.nseg_tgt; ++sg) a.xin[sg * seg + i] = xT;
  }
}

// Per-element arithmetic of the pixel samplers.  The single-purpose kernels below and the fused two-chain kernel call the same
// functions, so a value computed by the lock-step loop is the value the two-phase loops compute, bit for bit.
__device__ __forceinline__ float pixel_posterior_f(float x0, float xt, float nz, const cdx_pixel_coef& c) {
  if (c.ddpm) {
    const float mean = ADD(MUL(c.w0, x0), MUL(c.wt, xt));                                   // DW:293
    return ADD(mean, MUL(c.post_std, nz));                                                  // DW:297
  }
  const float et = DIV(SUB(xt, MUL(c.sqrt_at, x0)), c.sqrt_1m_at);                          // DW:299
  return ADD(ADD(MUL(c.sqrt_at_next, x0), MUL(c.c2, et)), MUL(c.c1, nz));                   // DW:302
}
__device__ __forceinline__ float pixel_eps_f(float xt, float xn, float et, const cdx_pixel_coef& c) {
  if (c.ddpm) {
    const float mean = MUL(c.inv_sqrt_1m_bt, SUB(xt, MUL(c.weight, et)));                   // DW:266
    return DIV(SUB(xn, mean), c.std_model);                                                 // DW:268
  }
  const float x0_t = DIV(SUB(xt, MUL(et, c.sqrt_1m_at)), c.sqrt_at);                        // DW:271
  return DIV(SUB(SUB(xn, MUL(c.sqrt_at_next, x0_t)), MUL(c.c2, et)), c.c1);                 // DW:275
}
__device__ __forceinline__ float pixel_step_f(float xt, float et, float nz, const cdx_pixel_coef& c) {
  if (c.ddpm) {
    const float mean = MUL(c.inv_sqrt_1m_bt, SUB(xt, MUL(c.weight, et)));                   // DW:204
    return ADD(mean, MUL(MUL(c.mask, c.std_model), nz));                                    // DW:208
  }
  const float x0_t = DIV(SUB(xt, MUL(et, c.sqrt_1m_at)), c.sqrt_at);                        // DW:213
  return ADD(ADD(MUL(c.sqrt_at_next, x0_t), MUL(c.c2, et)), MUL(c.c1, nz));                 // DW:222
}

__global__ void pixel_posterior_kernel(const float* __restrict__ x0, const float* __restrict__ xt, const float* __restrict__ nz,
                                       cdx_pixel_coef c, float* __restrict__ out, size_t n) {
  GRID_STRIDE(i, n) out[i] = pixel_posterior_f(x0[i], xt[i], nz[i], c);
}
__global__ void pixel_compute_eps_kernel(const float* __restrict__ xt, const float* __restrict__ xn, const float* __restrict__ et_,
                                         cdx_pixel_coef c, float* __restrict__ out, int B, int chw, int net_chw) {
  const size_t n = (size_t)B * chw;
  GRID_STRIDE(i, n) {
    const size_t b = i / chw;
    out[i] = pixel_eps_f(xt[i], xn[i], et_[b * net_chw + (i - b * chw)], c);
  }
}
__global__ void pixel_step_kernel(const float* __restrict__ xt, const float* __restrict__ et_, const float* __restrict__ eps,
                                  cdx_pixel_coef c, float* __restrict__ out, int B, int chw, int net_chw) {
  const size_t n = (size_t)B * chw;
  GRID_STRIDE(i, n) {
    const size_t b = i / chw;
    out[i] = pixel_step_f(xt[i], et_[b * net_chw + (i - b * chw)], eps ? eps[i] : 0.f, c);
  }
}
// One lock-step iteration of a two-model pixel cycle: the source chain's posterior sample, the noise it recovers from the source
// U-Net output, and the target chain's update with that noise.  The noise never leaves registers unless z_out asks for it.
__global__ void pixel_lock_step_kernel(const PixelLockStep a) {
  GRID_STRIDE(i, a.n) {
    const size_t b = i / a.chw, r = i - b * a.chw;
    const float xt = a.xt[i];
    const float xn = pixel_posterior_f(a.x0[i], xt, a.noise[i], a.cs);                       // sample_xt_next, DW:283-307
    const float eps = pixel_eps_f(xt, xn, a.et_src[b * a.net_chw_src + r], a.cs);             // compute_eps, DW:230-280
    a.x_next[i] = xn;
    if (a.z_out) a.z_out[b * a.z_stride + r] = eps;
    a.y_next[i] = pixel_step_f(a.y[i], a.et_tgt[b * a.net_chw_tgt + r], eps, a.ct);          // denoising_step_with_eps, DW:114-227
  }
}

}  // namespace

#define LAUNCH1(kernel, n, ...)                                   \
  do {                                                            \
    if (e.dry()) break;                                           \
    kernel<<<grid_for((n), e.num_sms), 256, 0, s>>>(__VA_ARGS__); \
    CDX_CUDA(cudaGetLastError());                                 \
    e.launches++;                                                 \
  } while (0)


// ------------------------------------------------------------------------------------------------ Directional-CLIP / metrics (8f-3)
// torch upsample_bicubic2d (aten/src/ATen/native/UpSample.h): A = -0.75, align_corners = False: src = (dst + 0.5) * scale - 0.5,
// 4 taps at floor(src) - 1 .. + 2 with clamped indices; weights from the cubic convolution polynomials.  Then (x - mean) / std.
__device__ __forceinline__ float cubic1(float x, float A) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; }
__device__ __forceinline__ float cubic2(float x, float A) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; }
__device__ __forceinline__ void cubic_coeffs(float t, float w[4]) {
  const float A = -0.75f;
  w[0] = cubic2(t + 1.f, A); w[1] = cubic1(t, A); w[2] = cubic1(1.f - t, A); w[3] = cubic2(2.f - t, A);
}
__global__ void clip_preprocess_kernel(const float* __restrict__ img, int B, int R, int size, float* __restrict__ out) {
  const float mean[3] = {0.48145466f, 0.4578275f, 0.40821073f}, sd[3] = {0.26862954f, 0.26130258f, 0.27577711f};   // clip.py _transform
  const float scale = (float)R / (float)size;
  const size_t n = (size_t)B * 3 * size * size;
  GRID_STRIDE(i, n) {
    const int x = (int)(i % size), y = (int)((i / size) % size), c = (int)((i / ((size_t)size * size)) % 3), b = (int)(i / ((size_t)3 * size * size));
    const float sy = ((float)y + 0.5f) * scale - 0.5f, sx = ((float)x + 0.5f) * scale - 0.5f;
    const float fy = floorf(sy), fx = floorf(sx);
    float wy[4], wx[4];
    cubic_coeffs(sy - fy, wy);
    cubic_coeffs(sx - fx, wx);
    const float* src = img + ((size_t)b * 3 + c) * R * R;
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int yy = min(max((int)fy - 1 + j, 0), R - 1);
      float row = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int xx = min(max((int)fx - 1 + k, 0), R - 1);
        row += src[(size_t)yy * R + xx] * wx[k];
      }
      acc += row * wy[j];
    }
    out[i] = (acc - mean[c]) / sd[c];
  }
}
// patch matrix for the stride-P patch embedding (conv P x P, stride P, no bias == GEMM): row = (b, py, px), col = (c, dy, dx)
__global__ void patchify_kernel(const float* __restrict__ img, float* __restrict__ out, int B, int S, int P) {
  const int np = S / P, K = 3 * P * P;
  const size_t n = (size_t)B * np * np * K;
  GRID_STRIDE(i, n) {
    const int col = (int)(i % K);
    const size_t row = i / K;
    const int px = (int)(row % np), py = (int)((row / np) % np), b = (int)(row / ((size_t)np * np));
    const int dx = col % P, dy = (col / P) % P, c = col / (P * P);
    out[i] = img[(((size_t)b * 3 + c) * S + (py * P + dy)) * S + px * P + dx];
  }
}
// x[b, 0] = class_embedding + pos[0]; x[b, 1 + i] = patch_i + pos[1 + i]      (CLIPVisionEmbeddings.forward)
__global__ void vit_tokens_kernel(const float* __restrict__ patches, const float* __restrict__ cls, const float* __restrict__ pos,
                                  float* __restrict__ out, int B, int N, int W) {
  const size_t n = (size_t)B * (N + 1) * W;
  GRID_STRIDE(i, n) {
    const int c = (int)(i % W);
    const int t = (int)((i / W) % (N + 1));
    const size_t b = i / ((size_t)(N + 1) * W);
    const float v = t == 0 ? cls[c] : patches[(b * N + (t - 1)) * W + c];
    out[i] = v + pos[(size_t)t * W + c];
  }
}
__global__ void gather_rows_kernel(const float* __restrict__ x, const int* __restrict__ rows, float* __restrict__ out, int B, int L, int W) {
  const size_t n = (size_t)B * W;
  GRID_STRIDE(i, n) {
    const size_t b = i / W;
    const int c = (int)(i - b * W);
    const int r = rows ? rows[b] : 0;
    out[i] = x[(b * L + r) * W + c];
  }
}
__global__ void eot_rows_kernel(const int* __restrict__ ids, int* __restrict__ rows, int B, int L) {      // text.argmax(dim=-1): first maximum
  GRID_STRIDE(b, (size_t)B) {
    int best = 0, bv = ids[b * L];
    for (int l = 1; l < L; ++l) {
      const int v = ids[b * L + l];
      if (v > bv) { bv = v; best = l; }
    }
    rows[b] = best;
  }
}
// one warp per sample
__global__ void dclip_scores_kernel(const float* __restrict__ img_f, const float* __restrict__ orig_f, const float* __restrict__ enc_f,
                                    const float* __restrict__ dec_f, int B, int D, float* __restrict__ clip_out, float* __restrict__ dclip_out) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  auto wsum = [&](float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
  };
  const float *pi = img_f + (size_t)b * D, *po = orig_f + (size_t)b * D, *pe = enc_f + (size_t)b * D, *pd = dec_f + (size_t)b * D;
  float si = 0.f, so = 0.f, se = 0.f, sd = 0.f;
  for (int c = lane; c < D; c += 32) { si += pi[c] * pi[c]; so += po[c] * po[c]; se += pe[c] * pe[c]; sd += pd[c] * pd[c]; }
  const float ni = sqrtf(wsum(si)), no = sqrtf(wsum(so)), ne = sqrtf(wsum(se)), nd = sqrtf(wsum(sd));
  float clip = 0.f, di2 = 0.f, dt2 = 0.f, dd = 0.f;
  for (int c = lane; c < D; c += 32) {
    const float a = pi[c] / ni, o = po[c] / no, e_ = pe[c] / ne, d = pd[c] / nd;
    clip += a * d;
    const float di = a - o, dt = d - e_;
    di2 += di * di; dt2 += dt * dt; dd += di * dt;
  }
  clip = wsum(clip); di2 = wsum(di2); dt2 = wsum(dt2); dd = wsum(dd);
  if (lane == 0) {
    clip_out[b] = clip;
    dclip_out[b] = dd / (sqrtf(di2) * sqrtf(dt2));         // <di / |di|, dt / |dt|>
  }
}
// PSNR / L2 partial sums (fp64) and SSIM over the valid region; grid = (tiles, B); out[b] = {sum sq diff, ssim sum over 3 channels}
__global__ void image_metrics_kernel(const float* __restrict__ a, const float* __restrict__ b_, int H, int W, double* __restrict__ acc) {
  const int img = blockIdx.y;
  const float* A = a + (size_t)img * 3 * H * W;
  const float* Bp = b_ + (size_t)img * 3 * H * W;
  __shared__ double gw[11];
  if (threadIdx.x == 0) {                 // cv2.getGaussianKernel(11, 1.5): exp(-(i-5)^2 / (2 sigma^2)), normalised
    double s = 0.0;
    for (int i = 0; i < 11; ++i) { gw[i] = exp(-((double)(i - 5) * (i - 5)) / (2.0 * 1.5 * 1.5)); s += gw[i]; }
    for (int i = 0; i < 11; ++i) gw[i] /= s;
  }
  __syncthreads();
  const int vh = H - 10, vw = W - 10;
  const size_t nvalid = (size_t)3 * vh * vw, npix = (size_t)3 * H * W;
  double sq = 0.0, ss = 0.0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += (size_t)gridDim.x * blockDim.x) {
    const float x = fminf(fmaxf(A[i], 0.f), 1.f), y = fminf(fmaxf(Bp[i], 0.f), 1.f);
    const float d = x - y;
    sq += (double)(d * d);                 // fp32 subtract / square as torch does, fp64 accumulation
  }
  const double C1 = (0.01 * 255) * (0.01 * 255), C2 = (0.03 * 255) * (0.03 * 255);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvalid; i += (size_t)gridDim.x * blockDim.x) {
    const int x = (int)(i % vw), y = (int)((i / vw) % vh), c = (int)(i / ((size_t)vw * vh));
    const float* pa = A + (size_t)c * H * W;
    const float* pb = Bp + (size_t)c * H * W;
    double m1 = 0, m2 = 0, s11 = 0, s22 = 0, s12 = 0;
    for (int dy = 0; dy < 11; ++dy) {
      for (int dx = 0; dx < 11; ++dx) {
        const double w = gw[dy] * gw[dx];
        // (img.numpy() * 255): fp32 product, then astype(float64)
        const double u = (double)(fminf(fmaxf(pa[(size_t)(y + dy) * W + x + dx], 0.f), 1.f) * 255.f);
        const double v = (double)(fminf(fmaxf(pb[(size_t)(y + dy) * W + x + dx], 0.f), 1.f) * 255.f);
        m1 += w * u; m2 += w * v; s11 += w * u * u; s22 += w * v * v; s12 += w * u * v;
      }
    }
    const double v1 = s11 - m1 * m1, v2 = s22 - m2 * m2, cv = s12 - m1 * m2;
    ss += ((2 * m1 * m2 + C1) * (2 * cv + C2)) / ((m1 * m1 + m2 * m2 + C1) * (v1 + v2 + C2));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { sq += __shfl_xor_sync(0xffffffffu, sq, o); ss += __shfl_xor_sync(0xffffffffu, ss, o); }
  if ((threadIdx.x & 31) == 0) { atomicAdd(acc + 2 * img, sq); atomicAdd(acc + 2 * img + 1, ss); }
}
__global__ void image_metrics_final_kernel(const double* __restrict__ acc, int B, int H, int W, float* __restrict__ out) {
  GRID_STRIDE(b, (size_t)B) {
    const double sq = acc[2 * b], ss = acc[2 * b + 1];
    const float mse = (float)(sq / ((double)3 * H * W));
    out[3 * b + 0] = mse == 0.f ? 100.f : 10.f * log10f(1.f / mse);
    out[3 * b + 1] = (float)(ss / ((double)3 * (H - 10) * (W - 10)));
    out[3 * b + 2] = sqrtf((float)sq);
  }
}

void latent_step(Engine& e, const LatentStep& a, cudaStream_t s) { LAUNCH1(latent_step_kernel, a.n, a); }
void latent_init(Engine& e, const LatentInit& a, cudaStream_t s) { LAUNCH1(latent_init_kernel, a.n, a); }
void affine(Engine& e, const float* x, float a, float b, float* out, size_t n, cudaStream_t s) { LAUNCH1(affine_kernel, n, x, a, b, out, n); }
void shift_scale(Engine& e, const float* x, float b, float a, float* out, size_t n, cudaStream_t s) { LAUNCH1(shift_scale_kernel, n, x, b, a, out, n); }
void q_sample(Engine& e, const float* x0, const float* nz, float sa, float s1, float* out, size_t n, cudaStream_t s) { LAUNCH1(q_sample_kernel, n, x0, nz, sa, s1, out, n); }
void silu(Engine& e, const float* x, float* y, size_t n, cudaStream_t s) { LAUNCH1(silu_kernel, n, x, y, n); }
void add(Engine& e, const float* a, const float* b, float* y, size_t n, cudaStream_t s) { LAUNCH1(add_kernel, n, a, b, y, n); }
void copy_rows(Engine& e, const float* a, float* y, size_t n, cudaStream_t s) { LAUNCH1(copy_kernel, n, a, y, n); }
void geglu(Engine& e, const float* x, float* y, int M, int C, cudaStream_t s, bool interleaved) {
  LAUNCH1(geglu_kernel, (size_t)M * C, x, y, (size_t)M, C, interleaved ? 1 : 0);
}
void interleave_geglu_rows(Engine& e, const float* src, float* dst, int rows, int rowlen, cudaStream_t s) {
  CDX_CHECK(rows % 128 == 0, "interleave_geglu_rows: %d rows", rows);
  LAUNCH1(interleave_geglu_rows_kernel, (size_t)rows * rowlen, src, dst, rows, rowlen);
}
void avgpool2(Engine& e, const float* x, float* y, int B, int H, int W, int C, cudaStream_t s) {
  CDX_CHECK(H % 2 == 0 && W % 2 == 0, "avgpool2: odd size %dx%d", H, W);
  LAUNCH1(avgpool2_kernel, (size_t)B * (H / 2) * (W / 2) * C, x, y, B, H, W, C);
}
void upsample2(Engine& e, const float* x, float* y, int B, int H, int W, int C, cudaStream_t s) {
  LAUNCH1(upsample2_kernel, (size_t)B * H * W * 4 * C, x, y, B, H, W, C);
}
void nchw_to_nhwc(Engine& e, const float* x, float* y, int B, int C, int HW, cudaStream_t s) {
  if (e.dry()) return;
  // x [b][C][HW] -> y [b][HW][C]
  transpose_kernel<<<dim3(cdiv(HW, 32), cdiv(C, 32), B), dim3(32, 8), 0, s>>>(x, y, C, HW);
  CDX_CUDA(cudaGetLastError());
  e.launches++;
}
void nhwc_to_nchw(Engine& e, const float* x, float* y, int B, int C, int HW, cudaStream_t s) {
  if (e.dry()) return;
  transpose_kernel<<<dim3(cdiv(C, 32), cdiv(HW, 32), B), dim3(32, 8), 0, s>>>(x, y, HW, C);
  CDX_CUDA(cudaGetLastError());
  e.launches++;
}
void timestep_embedding(Engine& e, const float* t, const float* freqs, float* emb, int B, int half, cudaStream_t s, bool sin_first) {
  if (e.dry()) return;
  temb_kernel<<<cdiv(B * half, 256), 256, 0, s>>>(t, freqs, emb, B, half, sin_first ? 1 : 0);
  CDX_CUDA(cudaGetLastError());
  e.launches++;
}
void repack_conv3x3(Engine& e, const float* w, float* o, int O, int I, cudaStream_t s, int Ipad) {
  const int Ip = Ipad > 0 ? Ipad : I;
  LAUNCH1(repack_conv_kernel, (size_t)O * Ip * 9, w, o, O, I, Ip);
}
void embed_tokens(Engine& e, const int* ids, const float* tok, const float* pos, float* out, int B, int L, int W, int vocab, cudaStream_t s) {
  LAUNCH1(embed_tokens_kernel, (size_t)B * L * W, ids, tok, pos, out, B, L, W, vocab);
}
void quick_gelu(Engine& e, const float* x, float* y, size_t n, cudaStream_t s) { LAUNCH1(quick_gelu_kernel, n, x, y, n); }
void gelu(Engine& e, const float* x, float* y, size_t n, cudaStream_t s) { LAUNCH1(gelu_kernel, n, x, y, n); }
void pad_channels(Engine& e, const float* x, float* y, size_t rows, int C, int Cp, cudaStream_t s) {
  LAUNCH1(pad_channels_kernel, rows * (size_t)Cp, x, y, rows, C, Cp);
}
void vae_posterior(Engine& e, const float* mom, const float* nz, float sf, float* out, int B, int C, int hw, cudaStream_t s) {
  LAUNCH1(vae_posterior_kernel, (size_t)B * C * hw, mom, nz, sf, out, B, C, hw);
}
void ddim_posterior_sample(Engine& e, const float* x0, const float* xt, const float* nz, const cdx_ddim_coef& c, float* out, size_t n, cudaStream_t s) {
  LAUNCH1(ddim_posterior_kernel, n, x0, xt, nz, c, out, n);
}
void ddim_compute_eps(Engine& e, const float* xt, const float* xn, const float* e_c, const float* e_uc, float scale, const cdx_ddim_coef& c,
                      float* out, size_t n, cudaStream_t s) {
  LAUNCH1(ddim_compute_eps_kernel, n, xt, xn, e_c, e_uc, scale, c, out, n);
}
void ddim_step_with_eps(Engine& e, const float* x, const float* e_c, const float* e_uc, float scale, const float* eps, const cdx_ddim_coef& c,
                        float* out, size_t n, cudaStream_t s) {
  LAUNCH1(ddim_step_kernel, n, x, e_c, e_uc, scale, eps, c, out, n);
}
void pixel_posterior_sample(Engine& e, const float* x0, const float* xt, const float* nz, const cdx_pixel_coef& c, float* out, size_t n, cudaStream_t s) {
  LAUNCH1(pixel_posterior_kernel, n, x0, xt, nz, c, out, n);
}
void pixel_compute_eps(Engine& e, const float* xt, const float* xn, const float* et, const cdx_pixel_coef& c, float* out, int B, int chw,
                       int net_chw, cudaStream_t s) {
  LAUNCH1(pixel_compute_eps_kernel, (size_t)B * chw, xt, xn, et, c, out, B, chw, net_chw);
}
void pixel_step_with_eps(Engine& e, const float* xt, const float* et, const float* eps, const cdx_pixel_coef& c, float* out, int B, int chw,
                         int net_chw, cudaStream_t s) {
  LAUNCH1(pixel_step_kernel, (size_t)B * chw, xt, et, eps, c, out, B, chw, net_chw);
}
void pixel_lock_step(Engine& e, const PixelLockStep& a, cudaStream_t s) { LAUNCH1(pixel_lock_step_kernel, a.n, a); }

// softmax(q k^T * scale) v through two batched contractions and a row softmax.  Scores live in the arena
// ([B*heads, Nq, ldS]); the fused tcgen05 flash kernel supersedes this when eligible.
void attention(Engine& e, const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, float* out, int ldo, int B, int Nq,
               int Nk, int heads, int d, int head_stride, float scale, cudaStream_t s, bool causal) {
  Scope sc(e.arena);
  const int ldS = (Nk + 3) & ~3;
  float* S = (float*)e.arena.alloc((size_t)B * heads * Nq * ldS * sizeof(float));
  GemmArgs g;
  g.M = Nq; g.N = Nk; g.K = d; g.mode = 0;
  g.A = q; g.lda = ldq; g.C1 = d;
  g.Bw = k; g.ldb = ldk; g.b_kn = 0;
  g.Cout = S; g.ldc = ldS; g.alpha = scale;
  g.batch = B; g.heads = heads;
  g.sA_b = (long long)Nq * ldq; g.sA_h = head_stride;
  g.sB_b = (long long)Nk * ldk; g.sB_h = head_stride;
  g.sC_b = (long long)heads * Nq * ldS; g.sC_h = (long long)Nq * ldS;
  gemm(e, g, s);
  softmax_rows(e, S, (long long)B * heads * Nq, Nk, ldS, s, causal ? Nq : 0);
  GemmArgs h;
  h.M = Nq; h.N = d; h.K = Nk; h.mode = 0;
  h.A = S; h.lda = ldS; h.C1 = Nk;
  h.Bw = v; h.ldb = ldv; h.b_kn = 1;
  h.Cout = out; h.ldc = ldo;
  h.batch = B; h.heads = heads;
  h.sA_b = (long long)heads * Nq * ldS; h.sA_h = (long long)Nq * ldS;
  h.sB_b = (long long)Nk * ldv; h.sB_h = head_stride;
  h.sC_b = (long long)Nq * ldo; h.sC_h = d;
  gemm(e, h, s);
}

}  // namespace cdx

namespace cdx {
namespace {
// one warp per latent pixel; lanes stride over the codebook, (distance, index) min-reduced with ties to the LOWER index (torch.argmin)
__global__ void vq_quantize_kernel(const float* __restrict__ z, const float* __restrict__ cb, float* __restrict__ out, size_t npix, int dim, int n_embed) {
  const size_t pix = (size_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (pix >= npix) return;
  const float* zp = z + pix * dim;
  float zz = 0.f;
  for (int c = 0; c < dim; ++c) zz += zp[c] * zp[c];
  float best = 3.4e38f;
  int bi = 0x7fffffff;
  for (int k = lane; k < n_embed; k += 32) {
    const float* e = cb + (size_t)k * dim;
    float ee = 0.f, dot = 0.f;
    for (int c = 0; c < dim; ++c) { ee += e[c] * e[c]; dot += zp[c] * e[c]; }
    const float d = (zz + ee) - 2.f * dot;
    if (d < best) { best = d; bi = k; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  for (int c = lane; c < dim; c += 32) out[pix * dim + c] = zp[c] + (cb[(size_t)bi * dim + c] - zp[c]);      // z + (z_q - z).detach()
}
}  // namespace
void vq_quantize(Engine& e, const float* z, const float* codebook, float* out, size_t npix, int dim, int n_embed, cudaStream_t s) {
  if (e.dry()) return;
  vq_quantize_kernel<<<(unsigned)((npix + 7) / 8), 256, 0, s>>>(z, codebook, out, npix, dim, n_embed);
  CDX_CUDA(cudaGetLastError());
  e.launches++;
}
void clip_preprocess(Engine& e, const float* img, int B, int R, int size, float* out, cudaStream_t s) {
  LAUNCH1(clip_preprocess_kernel, (size_t)B * 3 * size * size, img, B, R, size, out);
}
void patchify(Engine& e, const float* img, float* out, int B, int S, int P, cudaStream_t s) {
  LAUNCH1(patchify_kernel, (size_t)B * 3 * S * S, img, out, B, S, P);
}
void vit_tokens(Engine& e, const float* patches, const float* cls, const float* pos, float* out, int B, int N, int W, cudaStream_t s) {
  LAUNCH1(vit_tokens_kernel, (size_t)B * (N + 1) * W, patches, cls, pos, out, B, N, W);
}
void gather_rows(Engine& e, const float* x, const int* rows, float* out, int B, int L, int W, cudaStream_t s) {
  LAUNCH1(gather_rows_kernel, (size_t)B * W, x, rows, out, B, L, W);
}
void eot_rows(Engine& e, const int* ids, int* rows, int B, int L, cudaStream_t s) { LAUNCH1(eot_rows_kernel, (size_t)B, ids, rows, B, L); }
void dclip_scores(Engine& e, const float* img_f, const float* orig_f, const float* enc_f, const float* dec_f, int B, int D, float* clip_out,
                  float* dclip_out, cudaStream_t s) {
  if (e.dry()) return;
  dclip_scores_kernel<<<cdiv(B, 4), 128, 0, s>>>(img_f, orig_f, enc_f, dec_f, B, D, clip_out, dclip_out);
  CDX_CUDA(cudaGetLastError());
  e.launches++;
}
void image_metrics(Engine& e, const float* a, const float* b, int B, int H, int W, float* out, cudaStream_t s) {
  CDX_CHECK(H > 10 && W > 10, "image_metrics: %dx%d is smaller than the 11x11 SSIM window", H, W);
  Scope sc(e.arena);
  double* acc = (double*)e.arena.alloc((size_t)B * 2 * sizeof(double));
  if (e.dry()) return;
  CDX_CUDA(cudaMemsetAsync(acc, 0, (size_t)B * 2 * sizeof(double), s));
  const int tiles = std::min(e.num_sms * 4, cdiv((long long)3 * H * W, 256));
  image_metrics_kernel<<<dim3(tiles, B), 256, 0, s>>>(a, b, H, W, acc);
  CDX_CUDA(cudaGetLastError());
  e.launches++;
  LAUNCH1(image_metrics_final_kernel, (size_t)B, acc, B, H, W, out);
}
}  // namespace cdx
