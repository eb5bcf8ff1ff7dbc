// common.cuh -- engine-wide declarations: error plumbing, workspace arena, tensor views, op prototypes.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include <stdexcept>

#include "../../include/cdx.h"

namespace cdx {

// ------------------------------------------------------------------------------------------------
// errors: C++ exceptions inside the library, translated to CDX_E_* + thread-local message at the ABI
// ------------------------------------------------------------------------------------------------
struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
void set_last_error(const std::string& m);

#define CDX_CHECK(cond, ...)                                                     \
  do {                                                                           \
    if (!(cond)) {                                                               \
      char _b[512];                                                              \
      snprintf(_b, sizeof(_b), __VA_ARGS__);                                     \
      throw ::cdx::Error(CDX_E_INVALID, std::string(_b) + " [" #cond "]");       \
    }                                                                            \
  } while (0)

#define CDX_CUDA(expr)                                                                         \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      char _b[512];                                                                            \
      snprintf(_b, sizeof(_b), "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      throw ::cdx::Error(CDX_E_CUDA, _b);                                                      \
    }                                                                                          \
  } while (0)

// ------------------------------------------------------------------------------------------------
// workspace arena: stack (mark/release) allocator over one device slab, sized by a dry run of the call.
// All work of an engine is enqueued on a single stream, so memory released to the stack can be reused
// by later launches without extra synchronisation.
// ------------------------------------------------------------------------------------------------
struct Arena {
  char* base = nullptr;
  size_t cap = 0, off = 0, high = 0;
  bool dry = false;
  void* alloc(size_t bytes);
  size_t mark() const { return off; }
  void release(size_t m) { off = m; }
  void begin_dry();   // start a sizing pass: allocations only advance the offset
  void end_dry();     // grow the slab to the recorded high-water mark, rewind
  void destroy();
};

// per-kernel-family timing with CUDA events on the launching stream (bench.py's roofline numbers)
enum ProfTag {
  PROF_CONV_FFMA = 0, PROF_DENSE_FFMA = 1, PROF_BATCHED_FFMA = 2, PROF_CONV_TC = 3, PROF_DENSE_TC = 4, PROF_BATCHED_TC = 5,
  PROF_GROUPNORM = 6, PROF_LAYERNORM = 7, PROF_SOFTMAX = 8, PROF_ELEMENTWISE = 9, PROF_NTAGS = 10
};
struct ProfRec { cudaEvent_t a, b; int tag; double flops, bytes; int launches; char note[56]; };
struct Profiler {
  bool on = false;
  std::vector<ProfRec> recs;
  std::vector<cudaEvent_t> pool;
};

struct Engine {
  Profiler prof;
  int device = 0;
  int num_sms = 148;
  bool flash_attn = true;        // fused tcgen05 attention kernel (kernels_attn.cu); false -> unfused QK^T / softmax / PV
  int mma_mode = 1;              // 0 SIMT FFMA (exact fp32), 1 tcgen05
  int tc_kind = 1;               // tcgen05 product scheme: 0 3xTF32, 1 3x fp16-split at the kind::f16 rate (default), 2 1x fp16 (fast, not fp32-faithful)
  // tracked |max| scalars of activation tensors (operand range of the fp16-split GEMMs): a pool of device floats, handed out
  // per tensor by the graph executors and zeroed at the start of every network call
  float* amax_pool = nullptr;
  int amax_cap = 1 << 15, amax_used = 0, amax_high = 0;
  float* amax_slot();
  // per-(image, channel) fp64 statistics buffers of activation tensors (GroupNorm inputs), same life cycle as the amax slots
  double* stat_pool = nullptr;
  size_t stat_cap = (size_t)8 << 20, stat_used = 0, stat_high = 0;      // doubles (64 MB)
  double* stat_alloc(size_t n);
  void pools_reset(cudaStream_t s);   // start of a network call: zero what the previous call dirtied, rewind
  Arena arena;
  cudaStream_t last_stream = nullptr;   // stream of the previous arena-using call and the event recorded at its end
  cudaEvent_t done_ev = nullptr;
  bool ev_recorded = false;
  uint64_t launches = 0;
  cdx_gemm_plan last_gemm{};      // variant taken by the most recent GEMM's real pass (host only; read by the op-level test hook)
  bool dry() const { return arena.dry; }
};

// RAII: time everything enqueued between construction and destruction under one tag (no-op unless profiling)
struct ProfScope {
  Engine& e;
  cudaStream_t s;
  int idx = -1;
  ProfScope(Engine& eng, cudaStream_t st, int tag, double flops, double bytes, int launches);
  ~ProfScope();
  void note(const char* fmt, ...);     // free-form shape note, printed per launch when CDX_PROF_DUMP is set
};

struct Scope {   // RAII arena scope
  Arena& a;
  size_t m;
  explicit Scope(Arena& ar) : a(ar), m(ar.mark()) {}
  ~Scope() { a.release(m); }
};

// NHWC activation view: p[((b*H + y)*W + x)*C + c]; a [M,C] token matrix is H=M/B, W=1.
struct Tensor {
  float* p = nullptr;
  int B = 0, H = 0, W = 0, C = 0;
  float* amax = nullptr;      // device scalar >= max |element| (maintained by the producing kernel), or null when not tracked
  double* stats = nullptr;    // per-(image, channel) fp64 {sum, sum of squares} accumulated by the producing kernel, or null
  size_t numel() const { return (size_t)B * H * W * C; }
  int rows() const { return B * H * W; }
};
inline Tensor alloc_tensor(Engine& e, int B, int H, int W, int C) {
  Tensor t;
  t.B = B; t.H = H; t.W = W; t.C = C;
  t.p = (float*)e.arena.alloc(t.numel() * sizeof(float));
  return t;
}

// ------------------------------------------------------------------------------------------------
// dense contraction (implicit GEMM) arguments, shared by the SIMT and tcgen05 back ends
//   C[m,n] = alpha * sum_k A(m,k) * W(n,k)  (+ bias[n]) (+ rowvec[m / rows_per_batch, n]) (+ residual[m,n])
// A is either a dense row matrix (two channel-concatenated sources allowed) or the implicit im2col of
// a 3x3 convolution over an NHWC tensor (k = tap*Cin + c).
// ------------------------------------------------------------------------------------------------
struct GemmArgs {
  int M = 0, N = 0, K = 0;
  int mode = 0;                       // 0 dense rows, 1 conv3x3 gather
  const float* A = nullptr;  int lda = 0;  int C1 = 0;   // first source: C1 channels, row/pixel stride lda
  const float* A2 = nullptr; int lda2 = 0; int C2 = 0;   // optional second source (channel concat)
  // conv geometry (mode 1): stored input [B,Hin,Win,*], logical input is up x larger (nearest)
  int Hin = 0, Win = 0, Hout = 0, Wout = 0, stride = 1, pad = 1, up = 1;
  const float* Bw = nullptr; int ldb = 0; int b_kn = 0;   // weights [N][K] (b_kn=0) or [K][N] (b_kn=1)
  const float* Bw_hi = nullptr; const float* Bw_lo = nullptr;   // optional pre-split TF32 planes of Bw (same geometry)
  // optional fp16-split planes of Bw, pre-scaled by 2^b_exp (same geometry, element index = float index), and the tracked max |A|
  // scalars (device) of the A operand(s); c_amax: device scalar that receives max |C| (atomic max) for a consumer GEMM
  const void* Bw_h_hi = nullptr; const void* Bw_h_lo = nullptr; int b_exp = 0;
  const float* a_amax = nullptr; const float* a2_amax = nullptr;
  float* c_amax = nullptr;
  // conv3x3 halo schedule only: the A operand is silu?(x * a + o) with the per-(image, channel) table gn_ab [B, C1+C2] of float2 --
  // GroupNorm (+SiLU) of the input applied while the halo is converted; padding pixels stay exactly 0 (the reference pads the
  // normalised tensor).  A2 / C2: second source of a channel concat (C1 % 64 == 0)
  const float* gn_ab = nullptr; int gn_silu = 0;
  double* c_stats = nullptr;         // optional: += per-(image, channel) {sum, sum sq} of C (rows_per_batch rows per image), zeroed by the caller
  float* Cout = nullptr; int ldc = 0;
  float* Cout_lo = nullptr;           // if set: Cout receives rn_tf32(C) and Cout_lo rn_tf32(C - hi) (operand planes for tcgen05)
  // optional: columns n >= t_col0 are stored TRANSPOSED as TF32 planes, Ct_hi / Ct_lo [(n - t_col0) * ldt + m] (dense mode,
  // no split-K): the value projection of a fused q|k|v GEMM lands directly as the K-major V^T operand of the attention kernel
  float* Ct_hi = nullptr; float* Ct_lo = nullptr; int t_col0 = 0; long long ldt = 0;
  const float* bias = nullptr;
  const float* rowvec = nullptr; int ld_rowvec = 0; int rows_per_batch = 1;
  const float* residual = nullptr; int ldr = 0;
  float alpha = 1.f;
  int geglu = 0;                     // columns are [32 value | 32 gate] blocks: store value * gelu(gate) as [M, N/2] (attention.py:42-44)
  int out_nchw = 0;                  // store C as [B, N, rows_per_img] instead of [M, N]
  int rows_per_img = 0;
  // batching over blockIdx.z = zb*heads + zh
  int batch = 1, heads = 1;
  long long sA_b = 0, sA_h = 0, sB_b = 0, sB_h = 0, sC_b = 0, sC_h = 0;
};
void gemm(Engine& e, const GemmArgs& a, cudaStream_t s);
// tcgen05 back end (kernels_tc.cu); returns false when the shape is not eligible
bool gemm_tc(Engine& e, const GemmArgs& a, cudaStream_t s, int* side_done = nullptr);   // side_done bit 0: c_amax fused, bit 1: c_stats fused
bool flash_attention_tc(Engine& e, const float* q_hi, const float* q_lo, int ldq, const float* k_hi, const float* k_lo, int ldk,
                        const float* vt_hi, const float* vt_lo, float* out, int ldo, int B, int N, int Nk, int Nks, int heads, int d,
                        float scale, cudaStream_t s);
// fp16-split operands (the default scheme): planes made by split_rows_h16 / split_transpose_h16 from fp32 q | k and v with the
// tensors' tracked ranges (device slots); halves the tensor-pipe time and the operand bytes of the TF32-plane version
bool flash_attention_h16(Engine& e, const void* q_hi, const void* q_lo, int ldq, const void* k_hi, const void* k_lo, int ldk, const void* vt_hi,
                         const void* vt_lo, const float* q_amax, const float* k_amax, const float* v_amax, float* out, int ldo, int B, int N,
                         int Nk, int Nks, int heads, int d, float scale, cudaStream_t s);
void split_rows_h16(Engine& e, const float* src, long long rows, int cols, long long ld, void* hi, void* lo, long long ldh, const float* amax,
                    cudaStream_t s);
void split_transpose_h16(Engine& e, const float* src, int R, int Cc, long long ld, void* hi, void* lo, const float* amax, cudaStream_t s);
void split_planes(Engine& e, const float* w, float* hi, float* lo, size_t n, cudaStream_t s);   // hi = rn_tf32(w), lo = rn_tf32(w - hi)
// fp16 split of w * 2^exp: hi = fp16(w'), lo = fp16(w' - hi)  (hi / lo: __half arrays)
void split_planes_h16(Engine& e, const float* w, void* hi, void* lo, size_t n, int exp, cudaStream_t s);
// slot <- max(slot, max |x[r, 0..C)|) over `rows` rows of stride ld (atomic max on the bit pattern)
void amax_rows(Engine& e, const float* x, long long rows, int C, long long ld, float* slot, cudaStream_t s);
int h16_exp_host(float amax);   // exponent e with amax * 2^e in [2^14, 2^15)
bool attention_tc(Engine& e, const float* q, int ldq, const float* k, int ldk, int head_stride, const float* vt, float* out, int ldo, int B,
                  int Nq, int Nk, int heads, int d, float scale, cudaStream_t s);

// ------------------------------------------------------------------------------------------------
// normalisation / softmax / elementwise ops (kernels_norm.cu, kernels_elem.cu)
// ------------------------------------------------------------------------------------------------
// GroupNorm(32) over NHWC, optionally over the channel-concat of two sources; y = [silu]( gn(x)*(1+scale)+shift )
// st1 / st2: per-(image, channel) fp64 {sum, sum of squares} of the sources when their producer already accumulated them
// (stats[(b*C + c)*2 + k]); null -> computed here by one extra read.  amax: optional device scalar <- atomic max |y|.
void groupnorm(Engine& e, const float* x1, int C1, const float* x2, int C2, const float* gamma, const float* beta,
               float eps, bool silu, const float* scale, const float* shift, int ld_ss, float* y, int B, int HW,
               cudaStream_t s, const double* st1 = nullptr, const double* st2 = nullptr, float* amax = nullptr);
// the GroupNorm's per-(image, channel) affine table [B, C1+C2] of (a, o), y = x*a + o, for a conv that applies norm (+SiLU) itself
const float* gn_affine(Engine& e, const float* x1, int C1, const float* x2, int C2, const float* gamma, const float* beta, float eps,
                       const float* scale, const float* shift, int ld_ss, int B, int HW, cudaStream_t s, const double* st1, const double* st2);
// can a stride-1 conv3x3 over [B,H,W,C1(+C2)] take the halo schedule (and with it a fused GroupNorm + SiLU of its input)?
bool conv_halo_eligible(const Engine& e, int B, int H, int W, int C1, int C2, int Cout, bool out_nchw);
double* gn_channel_stats(Engine& e, const float* x, int C, int B, int HW, cudaStream_t s);
void gn_channel_stats_into(Engine& e, const float* x, int C, int B, int HW, double* stats, cudaStream_t s);   // stats += (zeroed by the caller)
void layernorm(Engine& e, const float* x, const float* gamma, const float* beta, float* y, int M, int C, cudaStream_t s, float* amax = nullptr);
// in place; causal_nq > 0: row r may only see columns j <= r % causal_nq (the rest become 0)
void softmax_rows(Engine& e, float* x, long long rows, int L, int ld, cudaStream_t s, int causal_nq = 0);
void silu(Engine& e, const float* x, float* y, size_t n, cudaStream_t s);
// x [M,2C] -> y [M,C] = value * gelu(gate); plain: value = x[:, :C], gate = x[:, C:]; interleaved: blocks of [32 value | 32 gate]
void geglu(Engine& e, const float* x, float* y, int M, int C, cudaStream_t s, bool interleaved = false);
void interleave_geglu_rows(Engine& e, const float* src, float* dst, int rows, int rowlen, cudaStream_t s);
void add(Engine& e, const float* a, const float* b, float* y, size_t n, cudaStream_t s);
void avgpool2(Engine& e, const float* x, float* y, int B, int H, int W, int C, cudaStream_t s);      // -> [B,H/2,W/2,C]
void upsample2(Engine& e, const float* x, float* y, int B, int H, int W, int C, cudaStream_t s);     // -> [B,2H,2W,C]
void nchw_to_nhwc(Engine& e, const float* x, float* y, int B, int C, int HW, cudaStream_t s);
void nhwc_to_nchw(Engine& e, const float* x, float* y, int B, int C, int HW, cudaStream_t s);
void timestep_embedding(Engine& e, const float* t, const float* freqs, float* emb, int B, int half, cudaStream_t s, bool sin_first = false);
void repack_conv3x3(Engine& e, const float* w, float* o, int O, int I, cudaStream_t s, int Ipad = 0);   // OIHW -> O,kh,kw,I (I zero-padded to Ipad)
void pad_channels(Engine& e, const float* x, float* y, size_t rows, int C, int Cp, cudaStream_t s);
void embed_tokens(Engine& e, const int* ids, const float* tok, const float* pos, float* out, int B, int L, int W, int vocab, cudaStream_t s);
void quick_gelu(Engine& e, const float* x, float* y, size_t n, cudaStream_t s);     // x * sigmoid(1.702 x)
void gelu(Engine& e, const float* x, float* y, size_t n, cudaStream_t s);           // exact erf GELU     // [rows,C] -> [rows,Cp], zero fill
void copy_rows(Engine& e, const float* src, float* dst, size_t n, cudaStream_t s);
// taming VectorQuantizer2.forward on NHWC latents: per pixel the first argmin_k of (|z|^2 + |e_k|^2) - 2 z.e_k, output z + (e_k - z)
void vq_quantize(Engine& e, const float* z, const float* codebook, float* out, size_t npix, int dim, int n_embed, cudaStream_t s);
// ---- Directional-CLIP / metric kernels (kernels_elem.cu; SURVEY 8f-3)
void clip_preprocess(Engine& e, const float* img, int B, int R, int size, float* out, cudaStream_t s);
void patchify(Engine& e, const float* img, float* out, int B, int S, int P, cudaStream_t s);            // [B,3,S,S] -> [B*(S/P)^2, 3*P*P]
void vit_tokens(Engine& e, const float* patches, const float* cls, const float* pos, float* out, int B, int N, int W, cudaStream_t s);
void gather_rows(Engine& e, const float* x, const int* row_of_batch, float* out, int B, int L, int W, cudaStream_t s);   // out[b] = x[b, row[b]]
void eot_rows(Engine& e, const int* ids, int* rows, int B, int L, cudaStream_t s);                      // first argmax of ids per sample
void dclip_scores(Engine& e, const float* img_f, const float* orig_f, const float* enc_f, const float* dec_f, int B, int D, float* clip_out,
                  float* dclip_out, cudaStream_t s);
void image_metrics(Engine& e, const float* a, const float* b, int B, int H, int W, float* out, cudaStream_t s);
void attention(Engine& e, const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, float* out, int ldo,
               int B, int Nq, int Nk, int heads, int d, int head_stride, float scale, cudaStream_t s, bool causal = false);

// scheduler kernels (kernels_elem.cu)
void affine(Engine& e, const float* x, float a, float b, float* out, size_t n, cudaStream_t s);
void shift_scale(Engine& e, const float* x, float b, float a, float* out, size_t n, cudaStream_t s);
void q_sample(Engine& e, const float* x0, const float* noise, float sa, float s1ma, float* out, size_t n, cudaStream_t s);
void vae_posterior(Engine& e, const float* moments, const float* noise, float sf, float* out, int B, int C, int hw, cudaStream_t s);
void ddim_posterior_sample(Engine& e, const float* x0, const float* xt, const float* noise, const cdx_ddim_coef& c, float* out, size_t n, cudaStream_t s);
void ddim_compute_eps(Engine& e, const float* xt, const float* xt_next, const float* e_c, const float* e_uc, float scale,
                      const cdx_ddim_coef& c, float* out, size_t n, cudaStream_t s);
void ddim_step_with_eps(Engine& e, const float* x, const float* e_c, const float* e_uc, float scale, const float* eps,
                        const cdx_ddim_coef& c, float* out, size_t n, cudaStream_t s);
// One fused elementwise launch per sampling step of the latent loops (DPM-Encoder, decode, or both in lock-step): recovers the
// noise of step i from the U-Net output (compute_eps), draws the next posterior sample of the source chain (sample_xt_next),
// advances the target chain with the recovered noise (p_sample_ddim_with_eps) and writes the next U-Net input batch.  Op order
// inside is that of the three single-purpose kernels above (bit-exact against the reference formulas).
struct LatentStep {
  size_t n = 0; int chw = 0;                 // B*chw elements
  // --- source chain (enc != 0)
  int enc = 0;
  const float* x0 = nullptr; const float* xt = nullptr; const float* xn = nullptr;    // x_t and x_{t-1} (already drawn)
  const float* es_c = nullptr; const float* es_uc = nullptr; float s_scale = 1.f;     // eps-hat under the source condition
  const float* s_scale_v = nullptr; const float* t_scale_v = nullptr;   // optional per-sample guidance scales [B] (ensemble members batched
                                                                        // along B); scale 1 -> eps-hat(c) and 0 -> eps-hat(uc) EXACTLY,
                                                                        // as the reference's single-forward branches (ddim.py:550-551)
  cdx_ddim_coef cs{};
  float* z_out = nullptr; long long z_stride = 0;   // optional: eps -> z_out[b*z_stride + r]
  int next = 0;                              // 0 none, 1 posterior sample x_{t-2} from (x0, xn, noise_next), 2 x_{t-2} = x0 (index 0)
  const float* noise_next = nullptr; cdx_ddim_coef cnext{};
  float* xn2 = nullptr;
  // --- target chain (dec != 0)
  int dec = 0;
  const float* yt = nullptr; const float* et_c = nullptr; const float* et_uc = nullptr; float t_scale = 1.f;
  cdx_ddim_coef ct{};
  const float* eps_in = nullptr; long long eps_stride = 0;    // dec without enc: recovered noise read from z (or extra noise, stride chw)
  float* y_out = nullptr;
  // --- next U-Net input batch [nseg, B, chw]: segments [0, nseg_src) <- x_{t-1}, [nseg_src, nseg_src + nseg_tgt) <- y_{t-1}
  float* xin = nullptr; int nseg_src = 0, nseg_tgt = 0;
};
void latent_step(Engine& e, const LatentStep& a, cudaStream_t s);
// x_T = sqrt(a_T) x0 + sqrt(1 - a_T) noise0 (ddim.py:477-479) -> z slot 0 (optional), x_T buffer, y_T buffer (optional), first
// posterior sample x_{T-1} (next as in LatentStep) and the first U-Net input batch
struct LatentInit {
  size_t n = 0; int chw = 0;
  const float* x0 = nullptr; const float* noise0 = nullptr; float sa = 0.f, s1 = 0.f;
  float* z_out = nullptr; long long z_stride = 0;
  float* xt = nullptr; float* yt = nullptr;
  int next = 0; const float* noise_next = nullptr; cdx_ddim_coef cnext{}; float* xn = nullptr;
  float* xin = nullptr; int nseg_src = 0, nseg_tgt = 0;
};
void latent_init(Engine& e, const LatentInit& a, cudaStream_t s);

void pixel_posterior_sample(Engine& e, const float* x0, const float* xt, const float* noise, const cdx_pixel_coef& c, float* out, size_t n, cudaStream_t s);
void pixel_compute_eps(Engine& e, const float* xt, const float* xt_next, const float* et, const cdx_pixel_coef& c, float* out,
                       int B, int chw, int net_chw, cudaStream_t s);
void pixel_step_with_eps(Engine& e, const float* xt, const float* et, const float* eps, const cdx_pixel_coef& c, float* out,
                         int B, int chw, int net_chw, cudaStream_t s);
// One iteration of the two-model pixel cycle in one launch: x_next = sample_xt_next(x0, xt, noise) and
// eps = compute_eps(xt, x_next, et_src) under cs (source chain), y_next = denoising_step_with_eps(y, et_tgt, eps) under ct (target
// chain).  Same per-element arithmetic as the three kernels above.  U-Net outputs are [B, Cnet, H, W] of which the first C channels
// are used (learn_sigma split, DW:236-238): net_chw_* = Cnet * H * W of each chain's network.
struct PixelLockStep {
  size_t n = 0; int chw = 0;                 // B*chw elements
  cdx_pixel_coef cs{}, ct{};
  const float* x0 = nullptr; const float* xt = nullptr; const float* noise = nullptr; float* x_next = nullptr;
  const float* et_src = nullptr; int net_chw_src = 0;
  const float* y = nullptr; const float* et_tgt = nullptr; int net_chw_tgt = 0; float* y_next = nullptr;
  float* z_out = nullptr; long long z_stride = 0;   // optional: eps -> z_out[b*z_stride + r]
};
void pixel_lock_step(Engine& e, const PixelLockStep& a, cudaStream_t s);

inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

}  // namespace cdx
