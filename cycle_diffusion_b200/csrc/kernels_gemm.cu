// kernels_gemm.cu -- fp32 FFMA implicit-GEMM tiles (the exact-fp32 contraction back end).
//
// One kernel family serves every dense contraction of the path:
//   * conv3x3 (stride 1/2, symmetric or asymmetric zero padding, fused nearest-2x upsample gather, channel-concat of
//     two sources)                          -- ResBlock / Downsample / Upsample convs (OAI:163-275, 91-160; AEM:42-141)
//   * conv1x1 / Linear (optionally two-source)  -- skip convs, proj_in/out, q/k/v/out, FF (ATT:152-261)
//   * batched Q.K^T and P.V                  -- attention score / value contractions (ATT:180-191, IU:351-361, AEM:187-197)
// Layout: activations NHWC (= token-major [M, C]), weights [N][K] with K = tap*Cin + c.  128x128x16 or 64x64x16
// CTA tiles, 256 threads, 8x8 / 4x4 register micro-tiles, double-buffered shared memory, 128-bit global loads.
// The tcgen05 back end (kernels_tc.cu) replaces this for TMA-eligible shapes; this one is always correct.
#include "common.cuh"

namespace cdx {

namespace {

constexpr int BK = 16;

struct RowInfo {   // per-thread, per-A-row precomputed gather state
  int valid;       // m < M
  int b, oy, ox;   // conv: sample, output pixel
  long long off1, off2;   // dense: row offsets into A / A2
};

template <int BM, int BN, int MODE, bool BKN, int VEC>
__global__ void __launch_bounds__(256, 2) gemm_kernel(GemmArgs p) {
  constexpr int TM = BM / 16, TN = BN / 16;
  constexpr int RM = TM / 4, RN = TN / 4;
  constexpr int LDAS = BM + 4, LDBS = BN + 4;
  constexpr int A_IT = BM / 64, B_IT = BN / 64;
  __shared__ __align__(16) float As[2][BK][LDAS];
  __shared__ __align__(16) float Bs[2][BK][LDBS];

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;

  // batch offsets
  const int z = blockIdx.z;
  const int zb = z / p.heads, zh = z - zb * p.heads;
  const float* __restrict__ A = p.A + zb * p.sA_b + zh * p.sA_h;
  const float* __restrict__ A2 = p.A2;
  const float* __restrict__ Bw = p.Bw + zb * p.sB_b + zh * p.sB_h;
  float* __restrict__ C = p.Cout + zb * p.sC_b + zh * p.sC_h;

  const int Cin = p.C1 + p.C2;
  const int a_row_l = tid >> 2;        // 0..63
  const int a_kq = (tid & 3) * 4;      // 0,4,8,12

  RowInfo ri[A_IT];
#pragma unroll
  for (int it = 0; it < A_IT; ++it) {
    const int m = m0 + a_row_l + it * 64;
    ri[it].valid = m < p.M;
    const int mm = ri[it].valid ? m : 0;
    if (MODE == 1) {
      const int hw = p.Hout * p.Wout;
      const int b = mm / hw;
      const int r = mm - b * hw;
      ri[it].b = b;
      ri[it].oy = r / p.Wout;
      ri[it].ox = r - ri[it].oy * p.Wout;
      ri[it].off1 = ri[it].off2 = 0;
    } else {
      ri[it].b = ri[it].oy = ri[it].ox = 0;
      ri[it].off1 = (long long)mm * p.lda;
      ri[it].off2 = (long long)mm * p.lda2;
    }
  }

  auto a_elem_ptr = [&](const RowInfo& r, int k, bool& ok) -> const float* {
    // address of A(m, k); ok=false -> zero
    ok = r.valid && (k < p.K);
    if (!ok) return A;
    if (MODE == 1) {
      const int tap = k / Cin;
      const int c = k - tap * Cin;
      const int dy = tap / 3, dx = tap - dy * 3;
      const int iy = r.oy * p.stride + dy - p.pad;
      const int ix = r.ox * p.stride + dx - p.pad;
      if (iy < 0 || ix < 0 || iy >= p.Hin * p.up || ix >= p.Win * p.up) { ok = false; return A; }
      const long long pix = ((long long)r.b * p.Hin + (iy / p.up)) * p.Win + (ix / p.up);
      return (c < p.C1) ? (A + pix * p.lda + c) : (A2 + pix * p.lda2 + (c - p.C1));
    } else {
      return (k < p.C1) ? (A + r.off1 + k) : (A2 + r.off2 + (k - p.C1));
    }
  };

  float4 ra[A_IT], rb[B_IT];

  auto load_a = [&](int kt) {
    const int k = kt * BK + a_kq;
#pragma unroll
    for (int it = 0; it < A_IT; ++it) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (VEC == 4) {
        bool ok;
        const float* ptr = a_elem_ptr(ri[it], k, ok);
        if (ok) {
          v = *reinterpret_cast<const float4*>(ptr);
          if (k + 3 >= p.K) {   // K tail inside this vector
            if (k + 1 >= p.K) v.y = 0.f;
            if (k + 2 >= p.K) v.z = 0.f;
            v.w = 0.f;
          }
        }
      } else {
        bool ok;
        const float* q;
        q = a_elem_ptr(ri[it], k + 0, ok); if (ok) v.x = *q;
        q = a_elem_ptr(ri[it], k + 1, ok); if (ok) v.y = *q;
        q = a_elem_ptr(ri[it], k + 2, ok); if (ok) v.z = *q;
        q = a_elem_ptr(ri[it], k + 3, ok); if (ok) v.w = *q;
      }
      ra[it] = v;
    }
  };

  auto load_b = [&](int kt) {
    if (!BKN) {
      const int k = kt * BK + a_kq;
#pragma unroll
      for (int it = 0; it < B_IT; ++it) {
        const int n = n0 + a_row_l + it * 64;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (n < p.N && k < p.K) {
          const float* ptr = Bw + (long long)n * p.ldb + k;
          if (VEC == 4) {
            v = *reinterpret_cast<const float4*>(ptr);
            if (k + 3 >= p.K) {
              if (k + 1 >= p.K) v.y = 0.f;
              if (k + 2 >= p.K) v.z = 0.f;
              v.w = 0.f;
            }
          } else {
            v.x = ptr[0];
            if (k + 1 < p.K) v.y = ptr[1];
            if (k + 2 < p.K) v.z = ptr[2];
            if (k + 3 < p.K) v.w = ptr[3];
          }
        }
        rb[it] = v;
      }
    } else {
      constexpr int F4_PER_ROW = BN / 4;          // 32 or 16
      constexpr int ROWS_PER_PASS = 256 / F4_PER_ROW;   // 8 or 16
      const int kl = tid / F4_PER_ROW;
      const int n4 = (tid % F4_PER_ROW) * 4;
#pragma unroll
      for (int it = 0; it < B_IT; ++it) {
        const int k = kt * BK + kl + it * ROWS_PER_PASS;
        const int n = n0 + n4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k < p.K && n < p.N) {
          const float* ptr = Bw + (long long)k * p.ldb + n;
          if (VEC == 4 && n + 3 < p.N) {
            v = *reinterpret_cast<const float4*>(ptr);
          } else {
            v.x = ptr[0];
            if (n + 1 < p.N) v.y = ptr[1];
            if (n + 2 < p.N) v.z = ptr[2];
            if (n + 3 < p.N) v.w = ptr[3];
          }
        }
        rb[it] = v;
      }
    }
  };

  auto store_smem = [&](int buf) {
#pragma unroll
    for (int it = 0; it < A_IT; ++it) {
      const int r = a_row_l + it * 64;
      As[buf][a_kq + 0][r] = ra[it].x;
      As[buf][a_kq + 1][r] = ra[it].y;
      As[buf][a_kq + 2][r] = ra[it].z;
      As[buf][a_kq + 3][r] = ra[it].w;
    }
    if (!BKN) {
#pragma unroll
      for (int it = 0; it < B_IT; ++it) {
        const int r = a_row_l + it * 64;
        Bs[buf][a_kq + 0][r] = rb[it].x;
        Bs[buf][a_kq + 1][r] = rb[it].y;
        Bs[buf][a_kq + 2][r] = rb[it].z;
        Bs[buf][a_kq + 3][r] = rb[it].w;
      }
    } else {
      constexpr int F4_PER_ROW = BN / 4;
      constexpr int ROWS_PER_PASS = 256 / F4_PER_ROW;
      const int kl = tid / F4_PER_ROW;
      const int n4 = (tid % F4_PER_ROW) * 4;
#pragma unroll
      for (int it = 0; it < B_IT; ++it)
        *reinterpret_cast<float4*>(&Bs[buf][kl + it * ROWS_PER_PASS][n4]) = rb[it];
    }
  };

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  const int KT = (p.K + BK - 1) / BK;
  load_a(0);
  load_b(0);
  store_smem(0);
  __syncthreads();

  for (int kt = 0; kt < KT; ++kt) {
    const int buf = kt & 1;
    if (kt + 1 < KT) {
      load_a(kt + 1);
      load_b(kt + 1);
    }
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float a[TM], b[TN];
#pragma unroll
      for (int r = 0; r < RM; ++r) {
        const float4 v = *reinterpret_cast<const float4*>(&As[buf][kk][r * 64 + ty * 4]);
        a[r * 4 + 0] = v.x; a[r * 4 + 1] = v.y; a[r * 4 + 2] = v.z; a[r * 4 + 3] = v.w;
      }
#pragma unroll
      for (int c = 0; c < RN; ++c) {
        const float4 v = *reinterpret_cast<const float4*>(&Bs[buf][kk][c * 64 + tx * 4]);
        b[c * 4 + 0] = v.x; b[c * 4 + 1] = v.y; b[c * 4 + 2] = v.z; b[c * 4 + 3] = v.w;
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (kt + 1 < KT) {
      store_smem(buf ^ 1);
      __syncthreads();
    }
  }

  // ---------------------------------------------------------------- epilogue
  const bool vec_ok = (VEC == 4) && !p.out_nchw && ((p.ldc & 3) == 0) &&
                      (p.residual == nullptr || (p.ldr & 3) == 0) && (p.rowvec == nullptr || (p.ld_rowvec & 3) == 0);
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int m = m0 + (i >> 2) * 64 + ty * 4 + (i & 3);
    if (m >= p.M) continue;
    const float* rv = p.rowvec ? p.rowvec + (long long)(m / p.rows_per_batch) * p.ld_rowvec : nullptr;
    const float* rs = p.residual ? p.residual + (long long)m * p.ldr : nullptr;
#pragma unroll
    for (int c = 0; c < RN; ++c) {
      const int n = n0 + c * 64 + tx * 4;
      if (n >= p.N) continue;
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = p.alpha * acc[i][c * 4 + j];
      if (vec_ok && n + 3 < p.N) {
        if (p.bias) {
          const float4 t = *reinterpret_cast<const float4*>(p.bias + n);
          v[0] += t.x; v[1] += t.y; v[2] += t.z; v[3] += t.w;
        }
        if (rv) {
          const float4 t = *reinterpret_cast<const float4*>(rv + n);
          v[0] += t.x; v[1] += t.y; v[2] += t.z; v[3] += t.w;
        }
        if (rs) {
          const float4 t = *reinterpret_cast<const float4*>(rs + n);
          v[0] += t.x; v[1] += t.y; v[2] += t.z; v[3] += t.w;
        }
        *reinterpret_cast<float4*>(C + (long long)m * p.ldc + n) = make_float4(v[0], v[1], v[2], v[3]);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int nn = n + j;
          if (nn >= p.N) break;
          float o = v[j];
          if (p.bias) o += p.bias[nn];
          if (rv) o += rv[nn];
          if (rs) o += rs[nn];
          if (p.out_nchw) {
            const int b = m / p.rows_per_img;
            const int r = m - b * p.rows_per_img;
            C[((long long)b * p.N + nn) * p.rows_per_img + r] = o;
          } else {
            C[(long long)m * p.ldc + nn] = o;
          }
        }
      }
    }
  }
}

template <int BM, int BN, int MODE, bool BKN, int VEC>
void launch(const GemmArgs& a, cudaStream_t s) {
  dim3 grid(cdiv(a.M, BM), cdiv(a.N, BN), a.batch * a.heads);
  gemm_kernel<BM, BN, MODE, BKN, VEC><<<grid, 256, 0, s>>>(a);
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

// side outputs a caller may ask for (range / GroupNorm statistics of C): fused into the tensor-core epilogue when it can,
// otherwise produced here by one extra pass over C (small / ragged shapes, the FFMA back end, split-K)
static void gemm_side_outputs(Engine& e, const GemmArgs& a, bool amax_done, bool stats_done, cudaStream_t s) {
  if (a.out_nchw) return;
  if (a.c_amax && !amax_done) amax_rows(e, a.Cout, a.M, a.geglu ? a.N / 2 : a.N, a.ldc, a.c_amax, s);
  if (a.c_stats && !stats_done) {
    CDX_CHECK(a.ldc == a.N && a.rows_per_batch > 0 && a.M % a.rows_per_batch == 0, "gemm: statistics need a dense [B*HW, N] result");
    gn_channel_stats_into(e, a.Cout, a.N, a.M / a.rows_per_batch, a.rows_per_batch, a.c_stats, s);
  }
}

void gemm(Engine& e, const GemmArgs& a, cudaStream_t s) {
  CDX_CHECK(a.M > 0 && a.N > 0 && a.K > 0, "gemm: empty problem M=%d N=%d K=%d", a.M, a.N, a.K);
  CDX_CHECK(a.batch >= 1 && a.heads >= 1, "gemm: bad batch");
  if (a.mode == 1) CDX_CHECK(a.K == 9 * (a.C1 + a.C2), "conv3x3: K != 9*Cin");
  if (a.mode == 0) CDX_CHECK(a.K == a.C1 + a.C2, "dense: K != C1+C2");
  if (e.mma_mode == 1) {
    int done = 0;                                          // bit 0: c_amax written, bit 1: c_stats written
    if (gemm_tc(e, a, s, &done)) {                         // (handles the arena dry run itself: split-K workspace)
      gemm_side_outputs(e, a, done & 1, done & 2, s);
      return;
    }
  }
  CDX_CHECK(!a.gn_ab && !(a.mode == 1 && a.A2), "gemm: a fused-GroupNorm / concat conv3x3 reached the FFMA back end (M=%d N=%d): the caller must ask conv_halo_eligible()",
            a.M, a.N);
  if (a.c_amax || a.c_stats) {
    GemmArgs b = a;
    b.c_amax = nullptr; b.c_stats = nullptr;
    gemm(e, b, s);
    gemm_side_outputs(e, a, false, false, s);
    return;
  }
  CDX_CHECK(!a.Ct_hi, "gemm: transposed plane output is only available on the tensor-core path (caller must check eligibility)");
  if (a.geglu) {       // fused only in the tensor-core epilogue; here: plain GEMM into a temporary, then the GEGLU kernel
    CDX_CHECK(a.N % 128 == 0 && a.batch * a.heads == 1 && !a.out_nchw && !a.Cout_lo, "gemm: bad GEGLU problem");
    Scope sc(e.arena);
    float* tmp = (float*)e.arena.alloc((size_t)a.M * a.N * sizeof(float));
    if (e.dry()) return;
    GemmArgs b = a;
    b.geglu = 0;
    b.Cout = tmp; b.ldc = a.N;
    gemm(e, b, s);
    CDX_CHECK(a.ldc == a.N / 2, "gemm: GEGLU output must be dense [M, N/2]");
    geglu(e, tmp, a.Cout, a.M, a.N / 2, s, true);
    return;
  }
  if (e.dry()) return;
  if (a.Cout_lo) {     // plane outputs are produced by the tensor-core epilogue; here: exact GEMM, then split in place
    CDX_CHECK(a.ldc == a.N && a.batch * a.heads == 1 && !a.out_nchw, "gemm: plane output needs a dense [M,N] result");
    GemmArgs b = a;
    b.Cout_lo = nullptr;
    gemm(e, b, s);
    split_planes(e, a.Cout, a.Cout, a.Cout_lo, (size_t)a.M * a.N, s);
    return;
  }
  e.last_gemm = cdx_gemm_plan{CDX_GEMM_FFMA, 0, 0, 0, 1, 0, 0};
  const double zz = (double)a.batch * a.heads;
  ProfScope ps(e, s, a.batch * a.heads > 1 ? PROF_BATCHED_FFMA : (a.mode == 1 ? PROF_CONV_FFMA : PROF_DENSE_FFMA),
               2.0 * a.M * a.N * a.K * zz, 4.0 * zz * ((double)a.M * a.K / (a.mode == 1 ? 9 : 1) + (double)a.N * a.K + (double)a.M * a.N), 1);

  // 128-bit path eligibility: every float4 must be 16B aligned and must not straddle sources / taps
  bool vec = aligned16(a.A) && (a.lda % 4 == 0) && (a.C1 % 4 == 0) && aligned16(a.Bw) && (a.ldb % 4 == 0);
  if (a.A2) vec = vec && aligned16(a.A2) && (a.lda2 % 4 == 0) && (a.C2 % 4 == 0);
  if (a.batch * a.heads > 1)
    vec = vec && (a.sA_b % 4 == 0) && (a.sA_h % 4 == 0) && (a.sB_b % 4 == 0) && (a.sB_h % 4 == 0) &&
          (a.sC_b % 4 == 0) && (a.sC_h % 4 == 0);
  vec = vec && aligned16(a.Cout) && (a.bias == nullptr || aligned16(a.bias)) &&
        (a.residual == nullptr || aligned16(a.residual)) && (a.rowvec == nullptr || aligned16(a.rowvec));
  if (a.b_kn) CDX_CHECK(a.mode == 0, "b_kn only for dense mode");

  const long long ctas128 = (long long)cdiv(a.M, 128) * cdiv(a.N, 128) * a.batch * a.heads;
  const bool big = ctas128 >= 2LL * e.num_sms && a.N > 64;

#define CDX_LAUNCH(MODE, BKN, VEC)                                   \
  do {                                                               \
    if (big) launch<128, 128, MODE, BKN, VEC>(a, s);                 \
    else launch<64, 64, MODE, BKN, VEC>(a, s);                       \
  } while (0)

  if (a.mode == 1) {
    if (vec) CDX_LAUNCH(1, false, 4); else CDX_LAUNCH(1, false, 1);
  } else if (a.b_kn) {
    if (vec) CDX_LAUNCH(0, true, 4); else CDX_LAUNCH(0, true, 1);
  } else {
    if (vec) CDX_LAUNCH(0, false, 4); else CDX_LAUNCH(0, false, 1);
  }
#undef CDX_LAUNCH
  CDX_CUDA(cudaGetLastError());
  e.launches++;
}

}  // namespace cdx
