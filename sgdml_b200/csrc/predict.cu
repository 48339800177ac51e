// Path (b): batched analytic energy/force prediction (SURVEY.md section 8 rows a-P, a-PT,
// a-M) -- reference sgdml/predict.py:84-245 (_predict_wkr), predict.py:424-441 (permuted
// caches), predict.py:551-601 (set_alphas), predict.py:1286-1288 (output scaling),
// torchtools.py:877-1046 (_forward).
//
// B200 design (not a port of either reference engine):
//  * Permutations are applied to the QUERY, never to the model: with e = perm_p[d],
//      delta_p[d] = x[d] - X_m[perm_p[d]]  ==  q_p[e] - X_m[e],  q_p[e] = x[pinv_p[e]],
//    so query b becomes S "virtual rows" q_{b,p} and the model stays an (M, D) pair of
//    matrices Xc (centred descriptors) and JA (= R_d_desc_alpha).  The reference
//    materialises an (M*S, D) permuted cache on the CPU (predict.py:426-437) and a
//    (B, M*S, D) temporary on the GPU (torchtools.py:964-966).
//  * The sum over training points is two GEMM-shaped contractions around an elementwise
//    Matern-5/2 transform -- the same shape as attention -- and both run on the FP64
//    tensor pipe (mma.sync m8n8k4.f64, SASS DMMA; tcgen05 has no f64 kind):
//      GEMM1: S1 = Q Xc^T, S2 = Q JA^T                      (contraction over D)
//      n^2 = |q|^2 + |Xc_m|^2 - 2 S1,  a = S2 - Xc_m.JA_m,  c1, c2 = Matern factors
//      GEMM2: G = (sum_m c1) Q - C1 Xc - C2 JA             (contraction over M)
//    G (BQ x DP) lives in registers for the whole sweep over M; Xc/JA tiles arrive through
//    a double-buffered cp.async.bulk (TMA engine) + mbarrier pipeline from L2.
//  * A small finishing kernel folds the S virtual rows back (F_desc[d] = sum_p
//    G_p[perm_p[d]]), applies J_x^T (predict.py:240-243) and the std / c scaling.
#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "desc.cuh"
#include "hessian.cuh"
#include "solve.cuh"

namespace sgdml {

// ============================================================== tile configuration
template <int DP_, int BQ_, int BM_, int W1Q_, int W1M_, int W1K_, int W2Q_, int W2D_, int MINB_ = 1, int W2S_ = 1,
          int OB_ = 0>
struct PCfg {
  // OB = 1 (fused configurations, W1K == 1): C1 / C2 double-buffered over tiles, ONE CTA-wide barrier per tile --
  // GEMM2 of tile t and GEMM1 + transform of tile t + 1 share a barrier interval, so warps drift apart and the tensor
  // pipe sees DMMA work from one warp while another runs the Matern transform; the bulk copies of tile t + 1 are issued
  // right after the barrier of tile t (its stage was last read by GEMM2 of tile t - 1)
  static constexpr int OB = OB_;
  static_assert(OB_ == 0 || W1K_ == 1, "one-barrier form needs the transform on the accumulator fragments");
  static constexpr int W2S = W2S_;      // 2: GEMM2 split by operand (warps 0-3: C1*Xc, warps 4-7: C2*JA)
  static constexpr int MINB = MINB_;    // CTAs per SM the kernel is compiled for
  static constexpr int DP = DP_;        // padded descriptor size (multiple of 8)
  static constexpr int DS = DP_ + 4;    // row stride of Q / Xc / JA tiles (== 4 or 12 mod 16: conflict-free DMMA frags)
  static constexpr int BQ = BQ_;        // virtual query rows per CTA
  static constexpr int BM = BM_;        // training points per pipeline stage
  static constexpr int CS = BM_ + 4;    // row stride of the S/C tiles
  static constexpr int W1Q = W1Q_, W1M = W1M_, W1K = W1K_;  // GEMM1 warp grid (rows, cols, split-k)
  static constexpr int W2Q = W2Q_, W2D = W2D_;              // GEMM2 warp grid (rows, cols)
  static constexpr int NT = 256;
  static constexpr int TR1 = BQ / (8 * W1Q);
  static constexpr int TC1 = BM / (8 * W1M);
  static constexpr int KS1 = DP / 4 / W1K;  // k-steps per warp in GEMM1
  static constexpr int TR2 = BQ / (8 * W2Q);
  static constexpr int TD2 = DP / (8 * W2D);
  static constexpr int EPT = BQ * BM / NT;  // epilogue-1 elements per thread
  // a warp that owns a single 8 x 8 fragment of S1 / S2 runs two interleaved accumulation chains over k (summed in
  // registers before the transform): four independent DMMAs in flight per warp instead of two
  static constexpr int KI = (W1K_ == 1 && TR1 * TC1 == 1 && KS1 % 2 == 0) ? 2 : 1;
  static_assert(W1Q * W1M * W1K == 8 && W2Q * W2D * W2S == 8 && (W2S == 1 || W2S == 2), "8 warps");
  static_assert(W2S == 1 || W1K * 2 * BQ_ * (BM_ + 4) >= BQ_ * DP_, "combine scratch must fit in the S/C region");
  static_assert(BQ % (8 * W1Q) == 0 && BM % (8 * W1M) == 0 && (DP / 4) % W1K == 0, "GEMM1 tiling");
  static_assert(BQ % (8 * W2Q) == 0 && DP % (8 * W2D) == 0, "GEMM2 tiling");
  static_assert(BM == 8 || BM == 16 || BM == 32, "row reduction uses shuffles inside one warp");
  static_assert((BQ * BM) % NT == 0, "epilogue mapping");
  // shared memory carve-up (in doubles)
  static constexpr int OFF_Q = 0;
  static constexpr int OFF_X = OFF_Q + BQ * DS;           // [2][BM*DS]
  static constexpr int OFF_JA = OFF_X + 2 * BM * DS;      // [2][BM*DS]
  static constexpr int OFF_MM = OFF_JA + 2 * BM * DS;     // [2][BM]
  static constexpr int OFF_XJA = OFF_MM + 2 * BM;         // [2][BM]
  static constexpr int OFF_AE = OFF_XJA + 2 * BM;         // [2][BM] energy-constraint coefficients (zeros when unused)
  static constexpr int OFF_P = OFF_AE + 2 * BM;           // [W1K][2][BQ*CS]; set 0 becomes C1/C2
  static constexpr int OFF_QQ = OFF_P + (OB_ ? 2 : 1) * W1K * 2 * BQ * CS;
  static constexpr int OFF_CSUM = OFF_QQ + BQ;
  static constexpr int OFF_E = OFF_CSUM + BQ;
  static constexpr int OFF_BAR = OFF_E + BQ;              // 3 x uint64
  static constexpr int SMEM_DOUBLES = OFF_BAR + 4;
  static constexpr size_t SMEM_BYTES = (size_t)SMEM_DOUBLES * 8;
  static_assert(SMEM_BYTES <= 232448, "exceeds 227 KB of shared memory");
  static_assert((BM * DS * 8) % 16 == 0 && (BM * 8) % 16 == 0 && (BQ * 8) % 16 == 0, "bulk copy granularity");
};

struct PredictArgs {
  // model (device)
  const double* Xc;     // (Mpad, DS) centred descriptors, zero padded
  const double* JA;     // (Mpad, DS) R_d_desc_alpha, zero padded
  const double* mm;     // (Mpad) |Xc_m|^2
  const double* xja;    // (Mpad) Xc_m . JA_m
  const double* ae;     // (Mpad) alphas_E (use_E_cstr models, predict.py:219-229); zeros when use_ae == 0
  int use_ae;
  int D, M, S, Mpad;
  double sig;
  // queries: virtual rows (b, p) prepared by k_query_rows
  const double* Qg;     // (rows padded to BQ, DS)  q_{b,p}[e] = x_b[pinv_p[e]] - mu[e], zero padded
  const double* qqg;    // (rows padded to BQ)      |q_{b,p}|^2
  int64_t n_rows;       // B*S virtual rows
  int64_t n_rows_pad;   // rows rounded up to BQ (stride between the per-split output planes)
  int tiles_per_split;  // blockIdx.y handles training tiles [y*tps, (y+1)*tps): small batches split the sweep over M
  int bm;               // training points per tile that tiles_per_split is counted in (the model's BM; a kernel with a
                        // smaller tile converts)
  // outputs
  double* G;            // (n_rows, DP)
  double* Erow;         // (n_rows)
};

// ============================================================== Matern-5/2 factors
// exp(-t) for t >= 0: Cody-Waite reduction + degree-12 Taylor polynomial (|r| <= ln2/2, truncation
// 1.7e-16 relative) -- ~16 FP64-pipe instructions instead of the library exp's ~22; the FP64 pipe
// is the kernel's bottleneck, so the transform is kept as lean as the 1e-6 force bound allows.
__device__ __forceinline__ double exp_neg(double t) {
  t = fmin(t, 708.0);
  const double kf = rint(-t * 1.4426950408889634074);
  double r = fma(kf, -6.93147180369123816490e-01, -t);
  r = fma(kf, -1.90821492927058770002e-10, r);
  // Estrin evaluation (dependency depth 5 instead of 12: the transform is latency-sensitive)
  const double r2 = r * r;
  const double a0 = 1.0 + r;
  const double a1 = fma(1.66666666666666666667e-01, r, 0.5);
  const double a2 = fma(8.33333333333333333333e-03, r, 4.16666666666666666667e-02);
  const double a3 = fma(1.98412698412698412698e-04, r, 1.38888888888888888889e-03);
  const double a4 = fma(2.75573192239858906526e-06, r, 2.48015873015873015873e-05);
  const double a5 = fma(2.50521083854417187751e-08, r, 2.75573192239858906526e-07);
  const double r4 = r2 * r2;
  const double b0 = fma(a1, r2, a0);
  const double b1 = fma(a3, r2, a2);
  const double b2 = fma(a5, r2, a4);
  const double r8 = r4 * r4;
  const double d0 = fma(b1, r4, b0);
  const double d1 = fma(2.08767569878680989792e-09, r4, b2);  // 1/12! r^12 term
  const double pv = fma(d1, r8, d0);
  const long long k = (long long)kf;
  return pv * __longlong_as_double((k + 1023) << 52);
}

struct MaternK {
  double sig, sig_inv, k_base, k_c1;  // k_c1 = k_base * 5/sig
};
// x5 = 5 (|q|^2 + |x|^2 - 2 q.x) (may be slightly negative), a = delta . JA  ->  c1, c2
// (predict.py:204-213):  n = sqrt(x5) = sqrt5 |delta|, base = exp(-n/sig) 5/(3 sig^3),
// c1 = a base 5/sig, c2 = base (n + sig)
__device__ __forceinline__ void matern52(double x5, double a, const MaternK& k, double& c1, double& c2) {
  const double x = fmax(x5, 1e-300);   // n = 1e-150 stands in for 0: no branch, no 0 * inf
  const double nrm = x * rsqrt(x);
  const double e = exp_neg(nrm * k.sig_inv);
  c1 = a * (e * k.k_c1);
  c2 = (e * k.k_base) * (nrm + k.sig);
}
// the same with the energy-constraint terms of predict.py:219-229 for a training point with coefficient ae:
//   F_desc += ae c2 delta  (folded into c1: both multiply delta),  E += ae K_ee,
//   K_ee = (1 + (n/sig)(1 + n/(3 sig))) exp(-n/sig);  returns the energy term a c2 + ae K_ee
__device__ __forceinline__ double matern52_ecstr(double x5, double a, double ae, const MaternK& k, double& c1, double& c2) {
  const double x = fmax(x5, 1e-300);
  const double nrm = x * rsqrt(x);
  const double t = nrm * k.sig_inv;
  const double e = exp_neg(t);
  c2 = (e * k.k_base) * (nrm + k.sig);
  c1 = fma(ae, c2, a * (e * k.k_c1));
  const double kee = fma(t, fma(t, 1.0 / 3.0, 1.0), 1.0) * e;
  return fma(a, c2, ae * kee);
}

// ============================================================== main kernel
template <class C>
__global__ void __launch_bounds__(256, C::MINB) k_predict_main(const PredictArgs p) {
  extern __shared__ __align__(128) double smem[];
  double* Qs = smem + C::OFF_Q;
  double* Xs = smem + C::OFF_X;
  double* JAs = smem + C::OFF_JA;
  double* mms = smem + C::OFF_MM;
  double* xjas = smem + C::OFF_XJA;
  double* aes = smem + C::OFF_AE;
  double* Ps = smem + C::OFF_P;
  double* qq = smem + C::OFF_QQ;
  double* csum_s = smem + C::OFF_CSUM;
  double* E_s = smem + C::OFF_E;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::OFF_BAR);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int lr = lane >> 2, lc = lane & 3;  // fragment row / k (or col pair) index
  const int64_t r0 = (int64_t)blockIdx.x * C::BQ;
  const int t_begin = (int)blockIdx.y * p.tiles_per_split;
  const int n_tiles = min(p.Mpad / C::BM, t_begin + p.tiles_per_split);  // exclusive end of this CTA's range
  constexpr uint32_t STAGE_BYTES = (uint32_t)((2 * C::BM * C::DS + 3 * C::BM) * 8);

  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_init(&bars[2], 1);
    fence_mbar_init();
  }
  __syncthreads();

  auto issue_tile = [&](int t) {
    const int s = (t - t_begin) & 1;
    const int64_t m0 = (int64_t)t * C::BM;
    mbar_arrive_expect_tx(&bars[s], STAGE_BYTES);
    bulk_g2s(Xs + s * C::BM * C::DS, p.Xc + m0 * C::DS, C::BM * C::DS * 8, &bars[s]);
    bulk_g2s(JAs + s * C::BM * C::DS, p.JA + m0 * C::DS, C::BM * C::DS * 8, &bars[s]);
    bulk_g2s(mms + s * C::BM, p.mm + m0, C::BM * 8, &bars[s]);
    bulk_g2s(xjas + s * C::BM, p.xja + m0, C::BM * 8, &bars[s]);
    bulk_g2s(aes + s * C::BM, p.ae + m0, C::BM * 8, &bars[s]);
  };
  if (tid == 0) {
    // the Q tile (BQ prepared virtual rows, contiguous) and its row norms: two bulk copies
    mbar_arrive_expect_tx(&bars[2], (uint32_t)((C::BQ * C::DS + C::BQ) * 8));
    bulk_g2s(Qs, p.Qg + r0 * C::DS, C::BQ * C::DS * 8, &bars[2]);
    bulk_g2s(qq, p.qqg + r0, C::BQ * 8, &bars[2]);
    issue_tile(t_begin);
    if (!C::OB && t_begin + 1 < n_tiles) issue_tile(t_begin + 1);
  }
  if (tid < C::BQ) {
    csum_s[tid] = 0.0;
    E_s[tid] = 0.0;
  }
  __syncthreads();
  mbar_wait(&bars[2], 0);

  // GEMM1 warp coordinates
  const int w1k = warp % C::W1K;
  const int w1m = (warp / C::W1K) % C::W1M;
  const int w1q = warp / (C::W1K * C::W1M);
  const int row1 = w1q * (C::TR1 * 8);
  const int col1 = w1m * (C::TC1 * 8);
  const int k1 = w1k * C::KS1 * 4;
  // GEMM2 warp coordinates
  constexpr int W2G = C::W2Q * C::W2D;  // warps per operand group
  const int w2s = warp / W2G;           // 0: Xc (and JA when W2S == 1), 1: JA
  const int w2d = (warp % W2G) % C::W2D;
  const int w2q = (warp % W2G) / C::W2D;
  const int row2 = w2q * (C::TR2 * 8);
  const int dcol2 = w2d * (C::TD2 * 8);

  double accG[C::TR2][C::TD2][2];
#pragma unroll
  for (int i = 0; i < C::TR2; ++i)
#pragma unroll
    for (int j = 0; j < C::TD2; ++j) accG[i][j][0] = accG[i][j][1] = 0.0;

  // running row sums: split-k path -> per epilogue element; fused path -> per fragment row
  constexpr int NPART = (C::W1K > 1) ? C::EPT : C::TR1;
  double csum_part[NPART], E_part[NPART];
#pragma unroll
  for (int j = 0; j < NPART; ++j) csum_part[j] = E_part[j] = 0.0;

  MaternK mk;
  mk.sig = p.sig;
  mk.sig_inv = 1.0 / p.sig;
  mk.k_base = 5.0 / (3.0 * p.sig * p.sig * p.sig);  // predict.py:195 mat52_base_fact
  mk.k_c1 = mk.k_base * 5.0 / p.sig;                // ... times predict.py:196 diag_scale_fact

  double* C1s = Ps;
  double* C2s = Ps + C::BQ * C::CS;

  for (int t = t_begin; t < n_tiles; ++t) {
    const int s = (t - t_begin) & 1;
    if constexpr (C::OB) {
      C1s = Ps + s * 2 * C::BQ * C::CS;
      C2s = C1s + C::BQ * C::CS;
    }
    const double* Xt = Xs + s * C::BM * C::DS;
    const double* JAt = JAs + s * C::BM * C::DS;
    const double* mmt = mms + s * C::BM;
    const double* xjat = xjas + s * C::BM;
    const double* aet = aes + s * C::BM;
    mbar_wait(&bars[s], (uint32_t)(((t - t_begin) >> 1) & 1));
    // real training points in this tile: the zero-padded tail of the last tile is skipped
    // (whole 8-point fragment columns in GEMM1, whole 4-point k-steps in GEMM2)
    const int mvalid = min(C::BM, p.M - t * C::BM);

    // ---------------- GEMM1: S1 = Q Xc^T, S2 = Q JA^T (over this warp's k-range)
    {
      double a1[C::TR1][C::TC1][2], a2[C::TR1][C::TC1][2];
#pragma unroll
      for (int i = 0; i < C::TR1; ++i)
#pragma unroll
        for (int j = 0; j < C::TC1; ++j) a1[i][j][0] = a1[i][j][1] = a2[i][j][0] = a2[i][j][1] = 0.0;
      const double* qa = Qs + (row1 + lr) * C::DS + k1 + lc;
      const double* xb = Xt + (col1 + lr) * C::DS + k1 + lc;
      const double* jb = JAt + (col1 + lr) * C::DS + k1 + lc;
      if constexpr (C::KI == 2) {
        // one fragment per warp: even and odd k-steps accumulate into separate registers
        double b1[2] = {0.0, 0.0}, b2[2] = {0.0, 0.0};
        if (col1 < mvalid) {  // warp-uniform
#pragma unroll 2
          for (int ks = 0; ks < C::KS1; ks += 2) {
            const double fa0 = qa[ks * 4], fa1 = qa[ks * 4 + 4];
            const double fx0 = xb[ks * 4], fx1 = xb[ks * 4 + 4];
            const double fj0 = jb[ks * 4], fj1 = jb[ks * 4 + 4];
            dmma884(a1[0][0][0], a1[0][0][1], fa0, fx0);
            dmma884(a2[0][0][0], a2[0][0][1], fa0, fj0);
            dmma884(b1[0], b1[1], fa1, fx1);
            dmma884(b2[0], b2[1], fa1, fj1);
          }
        }
        a1[0][0][0] += b1[0];
        a1[0][0][1] += b1[1];
        a2[0][0][0] += b2[0];
        a2[0][0][1] += b2[1];
      } else {
#pragma unroll 2
        for (int ks = 0; ks < C::KS1; ++ks) {
          double fa[C::TR1], fx[C::TC1], fj[C::TC1];
#pragma unroll
          for (int i = 0; i < C::TR1; ++i) fa[i] = qa[i * 8 * C::DS + ks * 4];
#pragma unroll
          for (int j = 0; j < C::TC1; ++j) {
            fx[j] = xb[j * 8 * C::DS + ks * 4];
            fj[j] = jb[j * 8 * C::DS + ks * 4];
          }
#pragma unroll
          for (int j = 0; j < C::TC1; ++j) {
            if (col1 + j * 8 < mvalid) {  // warp-uniform
#pragma unroll
              for (int i = 0; i < C::TR1; ++i) {
                dmma884(a1[i][j][0], a1[i][j][1], fa[i], fx[j]);
                dmma884(a2[i][j][0], a2[i][j][1], fa[i], fj[j]);
              }
            }
          }
        }
      }
      if constexpr (C::W1K == 1) {
        // fused: Matern transform straight on the accumulator fragments (predict.py:199-217)
#pragma unroll
        for (int j = 0; j < C::TC1; ++j) {
          const int mc = col1 + j * 8 + 2 * lc;
          if (col1 + j * 8 < mvalid) {  // warp-uniform: fragment columns of real training points
            const double m5a = 5.0 * mmt[mc], m5b = 5.0 * mmt[mc + 1];
            const double xa = xjat[mc], xb2 = xjat[mc + 1];
#pragma unroll
            for (int i = 0; i < C::TR1; ++i) {
              const int r = row1 + i * 8 + lr;
              const double q5 = 5.0 * qq[r];
              double c1a_, c2a_, c1b_, c2b_;
              const double aa = a2[i][j][0] - xa, ab = a2[i][j][1] - xb2;
              if (p.use_ae) {  // warp-uniform: models with energy constraints in the kernel
                E_part[i] += matern52_ecstr(fma(-10.0, a1[i][j][0], q5 + m5a), aa, aet[mc], mk, c1a_, c2a_);
                E_part[i] += matern52_ecstr(fma(-10.0, a1[i][j][1], q5 + m5b), ab, aet[mc + 1], mk, c1b_, c2b_);
              } else {
                matern52(fma(-10.0, a1[i][j][0], q5 + m5a), aa, mk, c1a_, c2a_);
                matern52(fma(-10.0, a1[i][j][1], q5 + m5b), ab, mk, c1b_, c2b_);
                E_part[i] = fma(aa, c2a_, fma(ab, c2b_, E_part[i]));
              }
              csum_part[i] += c1a_ + c1b_;
              const int off = r * C::CS + mc;
              *reinterpret_cast<double2*>(C1s + off) = make_double2(c1a_, c1b_);
              *reinterpret_cast<double2*>(C2s + off) = make_double2(c2a_, c2b_);
            }
          }
        }
      } else {
        double* P1 = Ps + (w1k * 2 + 0) * C::BQ * C::CS;
        double* P2 = Ps + (w1k * 2 + 1) * C::BQ * C::CS;
#pragma unroll
        for (int i = 0; i < C::TR1; ++i)
#pragma unroll
          for (int j = 0; j < C::TC1; ++j) {
            const int off = (row1 + i * 8 + lr) * C::CS + col1 + j * 8 + 2 * lc;
            *reinterpret_cast<double2*>(P1 + off) = make_double2(a1[i][j][0], a1[i][j][1]);
            *reinterpret_cast<double2*>(P2 + off) = make_double2(a2[i][j][0], a2[i][j][1]);
          }
      }
    }
    __syncthreads();
    if constexpr (C::OB) {
      if (tid == 0 && t + 1 < n_tiles) issue_tile(t + 1);
    }

    if constexpr (C::W1K > 1) {
      // ---------------- split-k: sum the partials, Matern transform in place
#pragma unroll
      for (int j = 0; j < C::EPT; ++j) {
        const int e = tid + j * C::NT;
        const int r = e / C::BM, mc = e % C::BM;
        const int off = r * C::CS + mc;
        double s1 = Ps[off], s2 = Ps[C::BQ * C::CS + off];
#pragma unroll
        for (int wk = 1; wk < C::W1K; ++wk) {
          s1 += Ps[(wk * 2 + 0) * C::BQ * C::CS + off];
          s2 += Ps[(wk * 2 + 1) * C::BQ * C::CS + off];
        }
        const double a = s2 - xjat[mc];
        double c1, c2;
        if (p.use_ae) {
          E_part[j] += matern52_ecstr(fma(-10.0, s1, 5.0 * (qq[r] + mmt[mc])), a, aet[mc], mk, c1, c2);
        } else {
          matern52(fma(-10.0, s1, 5.0 * (qq[r] + mmt[mc])), a, mk, c1, c2);
          E_part[j] = fma(a, c2, E_part[j]);
        }
        csum_part[j] += c1;
        C1s[off] = c1;
        C2s[off] = c2;
      }
      __syncthreads();
    }

    // ---------------- GEMM2: accG += C1 Xc + C2 JA (contraction over the BM points)
    {
      const double* c1a = C1s + (row2 + lr) * C::CS + lc;
      const double* c2a = C2s + (row2 + lr) * C::CS + lc;
      const double* xb = Xt + lc * C::DS + dcol2 + lr;
      const double* jb = JAt + lc * C::DS + dcol2 + lr;
      const int ks_end = (mvalid + 3) >> 2;
      if constexpr (C::W2S == 1) {
#pragma unroll 2
        for (int ks = 0; ks < ks_end; ++ks) {
          double f1[C::TR2], f2[C::TR2], fx[C::TD2], fj[C::TD2];
#pragma unroll
          for (int i = 0; i < C::TR2; ++i) {
            f1[i] = c1a[i * 8 * C::CS + ks * 4];
            f2[i] = c2a[i * 8 * C::CS + ks * 4];
          }
#pragma unroll
          for (int j = 0; j < C::TD2; ++j) {
            fx[j] = xb[ks * 4 * C::DS + j * 8];
            fj[j] = jb[ks * 4 * C::DS + j * 8];
          }
#pragma unroll
          for (int i = 0; i < C::TR2; ++i)
#pragma unroll
            for (int j = 0; j < C::TD2; ++j) {
              dmma884(accG[i][j][0], accG[i][j][1], f1[i], fx[j]);
              dmma884(accG[i][j][0], accG[i][j][1], f2[i], fj[j]);
            }
        }
      } else {
        const double* ca = w2s ? c2a : c1a;
        const double* ob = w2s ? jb : xb;
#pragma unroll 2
        for (int ks = 0; ks < ks_end; ++ks) {
          double f[C::TR2], fo[C::TD2];
#pragma unroll
          for (int i = 0; i < C::TR2; ++i) f[i] = ca[i * 8 * C::CS + ks * 4];
#pragma unroll
          for (int j = 0; j < C::TD2; ++j) fo[j] = ob[ks * 4 * C::DS + j * 8];
#pragma unroll
          for (int i = 0; i < C::TR2; ++i)
#pragma unroll
            for (int j = 0; j < C::TD2; ++j) dmma884(accG[i][j][0], accG[i][j][1], f[i], fo[j]);
        }
      }
    }
    if constexpr (!C::OB) {
      __syncthreads();
      if (tid == 0 && t + 2 < n_tiles) issue_tile(t + 2);
    }
  }

  // ---- row sums csum[r] = sum_m c1, E[r] = sum_m a c2
  if constexpr (C::W1K > 1) {
#pragma unroll
    for (int j = 0; j < C::EPT; ++j) {
      double cs = csum_part[j], es = E_part[j];
#pragma unroll
      for (int o = C::BM / 2; o > 0; o >>= 1) {
        cs += __shfl_xor_sync(0xffffffffu, cs, o);
        es += __shfl_xor_sync(0xffffffffu, es, o);
      }
      const int e = tid + j * C::NT;
      if (e % C::BM == 0) {
        csum_s[e / C::BM] = cs;
        E_s[e / C::BM] = es;
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < C::TR1; ++i) {
      double cs = csum_part[i], es = E_part[i];
      cs += __shfl_xor_sync(0xffffffffu, cs, 1);
      es += __shfl_xor_sync(0xffffffffu, es, 1);
      cs += __shfl_xor_sync(0xffffffffu, cs, 2);
      es += __shfl_xor_sync(0xffffffffu, es, 2);
      if (lc == 0) {  // W1M warps share a row: csum_s / E_s were zeroed before the sweep
        atomicAdd(&csum_s[row1 + i * 8 + lr], cs);
        atomicAdd(&E_s[row1 + i * 8 + lr], es);
      }
    }
  }
  if constexpr (C::W2S == 2) {
    if constexpr (C::OB) __syncthreads();  // GEMM2 of the last tile still reads C1 / C2
    // the JA group parks its partial sums in the (now free) S/C region
    if (w2s == 1) {
#pragma unroll
      for (int i = 0; i < C::TR2; ++i)
#pragma unroll
        for (int j = 0; j < C::TD2; ++j)
          *reinterpret_cast<double2*>(Ps + (row2 + i * 8 + lr) * C::DP + dcol2 + j * 8 + 2 * lc) =
              make_double2(accG[i][j][0], accG[i][j][1]);
    }
  }
  __syncthreads();

  // ---- G = (sum_m c1) Q - (C1 Xc + C2 JA)
  if (C::W2S == 1 || w2s == 0) {
#pragma unroll
    for (int i = 0; i < C::TR2; ++i) {
      const int r = row2 + i * 8 + lr;
      const int64_t row = r0 + r;
      if (row < p.n_rows) {
        const double cs = csum_s[r];
#pragma unroll
        for (int j = 0; j < C::TD2; ++j) {
          const int col = dcol2 + j * 8 + 2 * lc;
          double g0 = cs * Qs[r * C::DS + col] - accG[i][j][0];
          double g1 = cs * Qs[r * C::DS + col + 1] - accG[i][j][1];
          if constexpr (C::W2S == 2) {
            const double2 o = *reinterpret_cast<const double2*>(Ps + r * C::DP + col);
            g0 -= o.x;
            g1 -= o.y;
          }
          *reinterpret_cast<double2*>(p.G + ((int64_t)blockIdx.y * p.n_rows_pad + row) * C::DP + col) =
              make_double2(g0, g1);
        }
      }
    }
  }
  if (tid < C::BQ && r0 + tid < p.n_rows) p.Erow[(int64_t)blockIdx.y * p.n_rows_pad + r0 + tid] = E_s[tid];
}

// ============================================================== main kernel, two-group ("ping-pong") form
// The sweep of k_predict_main alternates tensor-pipe phases (GEMM1, GEMM2) with phases that leave the pipe idle (the
// split-k reduction + Matern transform, two CTA-wide barriers per tile): measured 77 % DMMA-active at BASELINE config 2
// (profiles/r01_ncu_predict_aspirin.txt).  Here the 8 warps form TWO groups of 4 (one warp of each group per SM
// sub-partition) that own half of the virtual query rows each and synchronise only among themselves (named
// barriers).  Group 0 runs  GEMM1(t) | transform(t) | GEMM2(t);  group 1 runs the same loop rotated,
// GEMM2(t) GEMM1(t+1) | transform(t+1), so the transform / barrier phases of one group fall into the tensor phases of
// the other and the pipe always has a warp with DMMA work.  The X / JA stage of a tile is handed back by whichever
// warp finishes with it last (a shared-memory counter): that warp issues the bulk copies of tile t + 2 -- no
// dedicated producer, nobody waits.  Used for the configurations with split-k GEMM1 (D > 72).
template <class C>
struct PPCfg {
  static constexpr int NG = 2;                // groups
  static constexpr int GT = C::NT / NG;       // threads per group (128)
  static constexpr int BQG = C::BQ / NG;      // virtual query rows per group
  static constexpr int W1Q = C::W1Q / NG, W1M = C::W1M, W1K = C::W1K;  // GEMM1 warp grid inside a group
  static constexpr int W2Q = C::W2Q / NG, W2D = C::W2D;                // GEMM2 warp grid inside a group
  static_assert(C::W1K > 1 && C::W2S == 1 && C::W1Q % NG == 0 && C::W2Q % NG == 0, "split-k configurations only");
  static_assert(W1Q * W1M * W1K == 4 && W2Q * W2D == 4, "4 warps per group");
  static constexpr int TR1 = BQG / (8 * W1Q), TC1 = C::BM / (8 * W1M), KS1 = C::DP / 4 / W1K;
  static constexpr int TR2 = BQG / (8 * W2Q), TD2 = C::DP / (8 * W2D);
  static constexpr int EPT = BQG * C::BM / GT;
  static_assert(TR1 * 8 * W1Q == BQG && TR2 * 8 * W2Q == BQG && (BQG * C::BM) % GT == 0, "group tiling");
  // shared memory (doubles): Q | X[2] | JA[2] | mm[2] | xja[2] | ae[2] | P [NG][W1K][2][BQG*CS] | Cc [NG][2][BQG*CS] | qq | csum | E | bars | cnt
  static constexpr int OFF_Q = 0;
  static constexpr int OFF_X = OFF_Q + C::BQ * C::DS;
  static constexpr int OFF_JA = OFF_X + 2 * C::BM * C::DS;
  static constexpr int OFF_MM = OFF_JA + 2 * C::BM * C::DS;
  static constexpr int OFF_XJA = OFF_MM + 2 * C::BM;
  static constexpr int OFF_AE = OFF_XJA + 2 * C::BM;
  static constexpr int OFF_P = OFF_AE + 2 * C::BM;
  static constexpr int P_GROUP = W1K * 2 * BQG * C::CS;
  static constexpr int OFF_C = OFF_P + NG * P_GROUP;
  static constexpr int C_GROUP = 2 * BQG * C::CS;
  static constexpr int OFF_QQ = OFF_C + NG * C_GROUP;
  static constexpr int OFF_CSUM = OFF_QQ + C::BQ;
  static constexpr int OFF_E = OFF_CSUM + C::BQ;
  static constexpr int OFF_BAR = OFF_E + C::BQ;  // 3 x uint64 + 2 x int
  static constexpr int SMEM_DOUBLES = OFF_BAR + 6;
  static constexpr size_t SMEM_BYTES = (size_t)SMEM_DOUBLES * 8;
  static_assert(SMEM_BYTES <= 232448, "exceeds 227 KB of shared memory");
};

__device__ __forceinline__ void group_barrier(int group) {
  asm volatile("bar.sync %0, 128;" ::"r"(1 + group) : "memory");
}

template <class C>
__global__ void __launch_bounds__(256, 1) k_predict_main_pp(const PredictArgs p) {
  using G = PPCfg<C>;
  extern __shared__ __align__(128) double smem[];
  double* Qs = smem + G::OFF_Q;
  double* Xs = smem + G::OFF_X;
  double* JAs = smem + G::OFF_JA;
  double* mms = smem + G::OFF_MM;
  double* xjas = smem + G::OFF_XJA;
  double* aes = smem + G::OFF_AE;
  double* qq = smem + G::OFF_QQ;
  double* csum_s = smem + G::OFF_CSUM;
  double* E_s = smem + G::OFF_E;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + G::OFF_BAR);
  int* cnt = reinterpret_cast<int*>(smem + G::OFF_BAR + 3);  // [2] stage hand-back counters

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int group = warp >> 2, wg = warp & 3, gtid = tid & (G::GT - 1);
  const int lr = lane >> 2, lc = lane & 3;
  const int64_t r0 = (int64_t)blockIdx.x * C::BQ;
  const int t_begin = (int)blockIdx.y * p.tiles_per_split;
  const int n_tiles = min(p.Mpad / C::BM, t_begin + p.tiles_per_split);
  constexpr uint32_t STAGE_BYTES = (uint32_t)((2 * C::BM * C::DS + 3 * C::BM) * 8);
  double* Ps = smem + G::OFF_P + group * G::P_GROUP;   // this group's split-k partials
  double* C1s = smem + G::OFF_C + group * G::C_GROUP;  // this group's transformed coefficients
  double* C2s = C1s + G::BQG * C::CS;
  const int grow0 = group * G::BQG;                    // first row of this group inside the CTA's Q tile

  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_init(&bars[2], 1);
    cnt[0] = cnt[1] = 0;
    fence_mbar_init();
  }
  __syncthreads();

  auto issue_tile = [&](int t) {
    const int s = (t - t_begin) & 1;
    const int64_t m0 = (int64_t)t * C::BM;
    mbar_arrive_expect_tx(&bars[s], STAGE_BYTES);
    bulk_g2s(Xs + s * C::BM * C::DS, p.Xc + m0 * C::DS, C::BM * C::DS * 8, &bars[s]);
    bulk_g2s(JAs + s * C::BM * C::DS, p.JA + m0 * C::DS, C::BM * C::DS * 8, &bars[s]);
    bulk_g2s(mms + s * C::BM, p.mm + m0, C::BM * 8, &bars[s]);
    bulk_g2s(xjas + s * C::BM, p.xja + m0, C::BM * 8, &bars[s]);
    bulk_g2s(aes + s * C::BM, p.ae + m0, C::BM * 8, &bars[s]);
  };
  if (tid == 0) {
    mbar_arrive_expect_tx(&bars[2], (uint32_t)((C::BQ * C::DS + C::BQ) * 8));
    bulk_g2s(Qs, p.Qg + r0 * C::DS, C::BQ * C::DS * 8, &bars[2]);
    bulk_g2s(qq, p.qqg + r0, C::BQ * 8, &bars[2]);
    issue_tile(t_begin);
    if (t_begin + 1 < n_tiles) issue_tile(t_begin + 1);
  }
  if (tid < C::BQ) {
    csum_s[tid] = 0.0;
    E_s[tid] = 0.0;
  }
  __syncthreads();
  mbar_wait(&bars[2], 0);

  // warp coordinates inside the group
  const int w1k = wg % G::W1K;
  const int w1m = (wg / G::W1K) % G::W1M;
  const int w1q = wg / (G::W1K * G::W1M);
  const int row1 = w1q * (G::TR1 * 8);
  const int col1 = w1m * (G::TC1 * 8);
  const int k1 = w1k * G::KS1 * 4;
  const int w2d = wg % G::W2D;
  const int w2q = wg / G::W2D;
  const int row2 = w2q * (G::TR2 * 8);
  const int dcol2 = w2d * (G::TD2 * 8);

  double accG[G::TR2][G::TD2][2];
#pragma unroll
  for (int i = 0; i < G::TR2; ++i)
#pragma unroll
    for (int j = 0; j < G::TD2; ++j) accG[i][j][0] = accG[i][j][1] = 0.0;
  double csum_part[G::EPT], E_part[G::EPT];
#pragma unroll
  for (int j = 0; j < G::EPT; ++j) csum_part[j] = E_part[j] = 0.0;

  MaternK mk;
  mk.sig = p.sig;
  mk.sig_inv = 1.0 / p.sig;
  mk.k_base = 5.0 / (3.0 * p.sig * p.sig * p.sig);
  mk.k_c1 = mk.k_base * 5.0 / p.sig;

  auto wait_full = [&](int t) { mbar_wait(&bars[(t - t_begin) & 1], (uint32_t)(((t - t_begin) >> 1) & 1)); };

  // ---------------- GEMM1 of tile t: this warp's k-range of S1 = Q Xc^T, S2 = Q JA^T -> partials in Ps
  auto gemm1 = [&](int t) {
    const int s = (t - t_begin) & 1;
    const double* Xt = Xs + s * C::BM * C::DS;
    const double* JAt = JAs + s * C::BM * C::DS;
    const int mvalid = min(C::BM, p.M - t * C::BM);
    double a1[G::TR1][G::TC1][2], a2[G::TR1][G::TC1][2];
#pragma unroll
    for (int i = 0; i < G::TR1; ++i)
#pragma unroll
      for (int j = 0; j < G::TC1; ++j) a1[i][j][0] = a1[i][j][1] = a2[i][j][0] = a2[i][j][1] = 0.0;
    const double* qa = Qs + (grow0 + row1 + lr) * C::DS + k1 + lc;
    const double* xb = Xt + (col1 + lr) * C::DS + k1 + lc;
    const double* jb = JAt + (col1 + lr) * C::DS + k1 + lc;
#pragma unroll 2
    for (int ks = 0; ks < G::KS1; ++ks) {
      double fa[G::TR1], fx[G::TC1], fj[G::TC1];
#pragma unroll
      for (int i = 0; i < G::TR1; ++i) fa[i] = qa[i * 8 * C::DS + ks * 4];
#pragma unroll
      for (int j = 0; j < G::TC1; ++j) {
        fx[j] = xb[j * 8 * C::DS + ks * 4];
        fj[j] = jb[j * 8 * C::DS + ks * 4];
      }
#pragma unroll
      for (int j = 0; j < G::TC1; ++j) {
        if (col1 + j * 8 < mvalid) {  // warp-uniform
#pragma unroll
          for (int i = 0; i < G::TR1; ++i) {
            dmma884(a1[i][j][0], a1[i][j][1], fa[i], fx[j]);
            dmma884(a2[i][j][0], a2[i][j][1], fa[i], fj[j]);
          }
        }
      }
    }
    double* P1 = Ps + (w1k * 2 + 0) * G::BQG * C::CS;
    double* P2 = Ps + (w1k * 2 + 1) * G::BQG * C::CS;
#pragma unroll
    for (int i = 0; i < G::TR1; ++i)
#pragma unroll
      for (int j = 0; j < G::TC1; ++j) {
        const int off = (row1 + i * 8 + lr) * C::CS + col1 + j * 8 + 2 * lc;
        *reinterpret_cast<double2*>(P1 + off) = make_double2(a1[i][j][0], a1[i][j][1]);
        *reinterpret_cast<double2*>(P2 + off) = make_double2(a2[i][j][0], a2[i][j][1]);
      }
  };

  // ---------------- split-k sum + Matern transform of tile t: Ps -> C1s, C2s
  auto transform = [&](int t) {
    const int s = (t - t_begin) & 1;
    const double* mmt = mms + s * C::BM;
    const double* xjat = xjas + s * C::BM;
    const double* aet = aes + s * C::BM;
#pragma unroll
    for (int j = 0; j < G::EPT; ++j) {
      const int e = gtid + j * G::GT;
      const int r = e / C::BM, mc = e % C::BM;
      const int off = r * C::CS + mc;
      double s1 = Ps[off], s2 = Ps[G::BQG * C::CS + off];
#pragma unroll
      for (int wk = 1; wk < G::W1K; ++wk) {
        s1 += Ps[(wk * 2 + 0) * G::BQG * C::CS + off];
        s2 += Ps[(wk * 2 + 1) * G::BQG * C::CS + off];
      }
      const double a = s2 - xjat[mc];
      double c1, c2;
      if (p.use_ae) {
        E_part[j] += matern52_ecstr(fma(-10.0, s1, 5.0 * (qq[grow0 + r] + mmt[mc])), a, aet[mc], mk, c1, c2);
      } else {
        matern52(fma(-10.0, s1, 5.0 * (qq[grow0 + r] + mmt[mc])), a, mk, c1, c2);
        E_part[j] = fma(a, c2, E_part[j]);
      }
      if (mc >= p.M - t * C::BM) c1 = c2 = 0.0;  // zero-padded training points of the last tile (C is read unmasked)
      csum_part[j] += c1;
      C1s[off] = c1;
      C2s[off] = c2;
    }
  };

  // ---------------- GEMM2 of tile t: accG += C1 Xc + C2 JA, then hand the stage back
  auto gemm2 = [&](int t) {
    const int s = (t - t_begin) & 1;
    const double* Xt = Xs + s * C::BM * C::DS;
    const double* JAt = JAs + s * C::BM * C::DS;
    const int mvalid = min(C::BM, p.M - t * C::BM);
    const double* c1a = C1s + (row2 + lr) * C::CS + lc;
    const double* c2a = C2s + (row2 + lr) * C::CS + lc;
    const double* xb = Xt + lc * C::DS + dcol2 + lr;
    const double* jb = JAt + lc * C::DS + dcol2 + lr;
    const int ks_end = (mvalid + 3) >> 2;
#pragma unroll 2
    for (int ks = 0; ks < ks_end; ++ks) {
      double f1[G::TR2], f2[G::TR2], fx[G::TD2], fj[G::TD2];
#pragma unroll
      for (int i = 0; i < G::TR2; ++i) {
        f1[i] = c1a[i * 8 * C::CS + ks * 4];
        f2[i] = c2a[i * 8 * C::CS + ks * 4];
      }
#pragma unroll
      for (int j = 0; j < G::TD2; ++j) {
        fx[j] = xb[ks * 4 * C::DS + j * 8];
        fj[j] = jb[ks * 4 * C::DS + j * 8];
      }
#pragma unroll
      for (int i = 0; i < G::TR2; ++i)
#pragma unroll
        for (int j = 0; j < G::TD2; ++j) {
          dmma884(accG[i][j][0], accG[i][j][1], f1[i], fx[j]);
          dmma884(accG[i][j][0], accG[i][j][1], f2[i], fj[j]);
        }
    }
    // the last of the 8 warps to finish with this stage refills it with tile t + 2
    __syncwarp();
    if (lane == 0) {
      const int old = atomicAdd(&cnt[s], 1);
      if (old == 7) {
        atomicExch(&cnt[s], 0);
        if (t + 2 < n_tiles) issue_tile(t + 2);
      }
    }
  };

  if (group == 0) {
    for (int t = t_begin; t < n_tiles; ++t) {
      wait_full(t);
      gemm1(t);
      group_barrier(group);
      transform(t);
      group_barrier(group);
      gemm2(t);
    }
  } else {
    if (t_begin < n_tiles) {
      wait_full(t_begin);
      gemm1(t_begin);
      group_barrier(group);
      transform(t_begin);
      group_barrier(group);
    }
    for (int t = t_begin; t < n_tiles; ++t) {
      gemm2(t);
      if (t + 1 < n_tiles) {
        wait_full(t + 1);
        gemm1(t + 1);
        group_barrier(group);
        transform(t + 1);
        group_barrier(group);
      }
    }
  }

  // ---- row sums csum[r] = sum_m c1, E[r] = sum_m a c2 (fixed order: shuffles inside the BM-lane segments)
#pragma unroll
  for (int j = 0; j < G::EPT; ++j) {
    double cs = csum_part[j], es = E_part[j];
#pragma unroll
    for (int o = C::BM / 2; o > 0; o >>= 1) {
      cs += __shfl_xor_sync(0xffffffffu, cs, o);
      es += __shfl_xor_sync(0xffffffffu, es, o);
    }
    const int e = gtid + j * G::GT;
    if (e % C::BM == 0) {
      csum_s[grow0 + e / C::BM] = cs;
      E_s[grow0 + e / C::BM] = es;
    }
  }
  group_barrier(group);

  // ---- G = (sum_m c1) Q - (C1 Xc + C2 JA)
#pragma unroll
  for (int i = 0; i < G::TR2; ++i) {
    const int r = grow0 + row2 + i * 8 + lr;
    const int64_t row = r0 + r;
    if (row < p.n_rows) {
      const double cs = csum_s[r];
#pragma unroll
      for (int j = 0; j < G::TD2; ++j) {
        const int col = dcol2 + j * 8 + 2 * lc;
        const double g0 = cs * Qs[r * C::DS + col] - accG[i][j][0];
        const double g1 = cs * Qs[r * C::DS + col + 1] - accG[i][j][1];
        *reinterpret_cast<double2*>(p.G + ((int64_t)blockIdx.y * p.n_rows_pad + row) * C::DP + col) = make_double2(g0, g1);
      }
    }
  }
  if (gtid < G::BQG && r0 + grow0 + gtid < p.n_rows)
    p.Erow[(int64_t)blockIdx.y * p.n_rows_pad + r0 + grow0 + gtid] = E_s[grow0 + gtid];
}

// ============================================================== query rows
// One warp per virtual row (b, p): Qg[row][e] = x_b[pinv_p[e]] - mu[e] (zero beyond D and beyond the
// last real row, so that every main-kernel tile is one contiguous bulk copy) and qq[row] = |Qg[row]|^2.
__global__ void __launch_bounds__(256) k_query_rows(const double* __restrict__ xq, const int* __restrict__ pinv,
                                                    const double* __restrict__ mu, int D, int DS, int S,
                                                    int64_t n_rows, int64_t n_rows_pad, double* __restrict__ Qg,
                                                    double* __restrict__ qqg) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n_rows_pad) return;
  double s = 0.0;
  if (row < n_rows) {
    const int64_t b = row / S;
    const int pp = (int)(row - b * S);
    const double* x = xq + b * D;
    const int* pi = pinv + pp * D;
    for (int e = lane; e < DS; e += 32) {
      double v = 0.0;
      if (e < D) v = x[pi[e]] - mu[e];
      Qg[row * DS + e] = v;
      s = fma(v, v, s);
    }
  } else {
    for (int e = lane; e < DS; e += 32) Qg[row * DS + e] = 0.0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) qqg[row] = s;
}

// Small host-buffer batches (the CUDA-graph path): descriptor, its derivative factors and the S query rows of one
// geometry in ONE launch, one CTA per geometry.  R may live in pinned host memory (read once into shared memory through
// the unified address space); the arithmetic is that of k_desc_from_R (csrc/desc.cu) followed by k_query_rows.
__global__ void __launch_bounds__(256) k_desc_query_rows(const double* __restrict__ R, int n_atoms,
                                                         const int* __restrict__ pinv, const double* __restrict__ mu,
                                                         int D, int DS, int S, int64_t n_rows, int64_t n_rows_pad,
                                                         double* __restrict__ gq, double* __restrict__ Qg,
                                                         double* __restrict__ qqg, const Lattice lat) {
  extern __shared__ double dq_sm[];  // r: 3N, x: D
  double* r = dq_sm;
  double* x = dq_sm + 3 * n_atoms;
  const int64_t b = blockIdx.x;
  for (int i = threadIdx.x; i < 3 * n_atoms; i += blockDim.x) r[i] = R[b * 3 * n_atoms + i];
  __syncthreads();
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    int a, c;
    pair_from_d(d, a, c);
    double dx = r[3 * a + 0] - r[3 * c + 0];
    double dy = r[3 * a + 1] - r[3 * c + 1];
    double dz = r[3 * a + 2] - r[3 * c + 2];
    if (lat.on) {
      const double c0 = rint(lat.inv[0] * dx + lat.inv[1] * dy + lat.inv[2] * dz);
      const double c1 = rint(lat.inv[3] * dx + lat.inv[4] * dy + lat.inv[5] * dz);
      const double c2 = rint(lat.inv[6] * dx + lat.inv[7] * dy + lat.inv[8] * dz);
      dx -= lat.vec[0] * c0 + lat.vec[1] * c1 + lat.vec[2] * c2;
      dy -= lat.vec[3] * c0 + lat.vec[4] * c1 + lat.vec[5] * c2;
      dz -= lat.vec[6] * c0 + lat.vec[7] * c1 + lat.vec[8] * c2;
    }
    const double dist = sqrt(dx * dx + dy * dy + dz * dz);
    const double inv3 = 1.0 / (dist * dist * dist);
    x[d] = 1.0 / dist;
    double* g = gq + (b * D + d) * 3;
    g[0] = dx * inv3;
    g[1] = dy * inv3;
    g[2] = dz * inv3;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  // rows b*S .. b*S+S-1; the last CTA also clears the padding rows of the last main-kernel tile
  const int extra = b == (int64_t)gridDim.x - 1 ? (int)(n_rows_pad - n_rows) : 0;
  for (int pp = warp; pp < S + extra; pp += n_warps) {
    const int64_t row = b * S + pp;
    double s = 0.0;
    if (pp < S) {
      const int* pi = pinv + pp * D;
      for (int e = lane; e < DS; e += 32) {
        double v = 0.0;
        if (e < D) v = x[pi[e]] - mu[e];
        Qg[row * DS + e] = v;
        s = fma(v, v, s);
      }
    } else {
      for (int e = lane; e < DS; e += 32) Qg[row * DS + e] = 0.0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) qqg[row] = s;
  }
}

// ============================================================== large descriptors (D > 256)
// The accumulator tile G (BQ x DP) of the fused kernel no longer fits the register file, so the
// same four contractions run as plain DMMA GEMMs (csrc/solve.cu) around two element-wise kernels:
//   S1 = Q Xc^T, S2 = Q JA^T (GEMM, k = D) -> k_transform_rows (in place: S1 -> C1, S2 -> C2)
//   acc = C1 XcT^T + C2 JAT^T (GEMM, k = M)  -> k_combine_rows: G = (sum_m c1) Q - acc
// Per (row, m) pair this adds 64 B of HBM traffic to >= 9 * 256 flop: far above the FP64 ridge.
__global__ void __launch_bounds__(256) k_transform_rows(double* __restrict__ S1, double* __restrict__ S2, int64_t ldS,
                                                        const double* __restrict__ qq, const double* __restrict__ mm,
                                                        const double* __restrict__ xja,
                                                        const double* __restrict__ ae, int M, int Mpad,
                                                        int64_t n_rows, MaternK mk, double* __restrict__ csum,
                                                        double* __restrict__ Erow) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  double* s1 = S1 + r * ldS;
  double* s2 = S2 + r * ldS;
  const double q5 = 5.0 * qq[r];
  double cs = 0.0, es = 0.0;
  for (int m = lane; m < Mpad; m += 32) {
    double c1 = 0.0, c2 = 0.0;
    if (m < M) {
      const double a = s2[m] - xja[m];
      if (ae != nullptr) {
        es += matern52_ecstr(fma(-10.0, s1[m], q5 + 5.0 * mm[m]), a, ae[m], mk, c1, c2);
      } else {
        matern52(fma(-10.0, s1[m], q5 + 5.0 * mm[m]), a, mk, c1, c2);
        es = fma(a, c2, es);
      }
      cs += c1;
    }
    s1[m] = c1;
    s2[m] = c2;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    cs += __shfl_xor_sync(0xffffffffu, cs, o);
    es += __shfl_xor_sync(0xffffffffu, es, o);
  }
  if (lane == 0) {
    csum[r] = cs;
    Erow[r] = es;
  }
}

__global__ void k_combine_rows(const double* __restrict__ Qg, int64_t ldq, const double* __restrict__ csum,
                               double* __restrict__ G, int DP, int64_t n_rows) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_rows * DP) return;
  const int64_t r = idx / DP;
  const int d = (int)(idx - r * DP);
  G[idx] = csum[r] * Qg[r * ldq + d] - G[idx];
}

// src (rows x cols, lds) -> dst (cols x rows), ldd >= rows
__global__ void k_transpose_pad(const double* __restrict__ src, int64_t rows, int64_t cols, int64_t lds,
                                double* __restrict__ dst, int64_t ldd) {
  __shared__ double tile[32][33];
  const int64_t r0 = (int64_t)blockIdx.y * 32, c0 = (int64_t)blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? src[r * lds + c] : 0.0;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows) dst[c * ldd + r] = tile[threadIdx.x][i];
  }
}

// ============================================================== finishing kernel
// F_desc[d] = sum_p G[b*S+p][perm_p[d]];  F = J_x^T F_desc (predict.py:240-243);
// E = sum_p Erow;  outputs scaled by std, E += c (predict.py:1286-1288).
// One CTA per QPB queries (QPB = 128 / D for small molecules, else 1): threads over (query, descriptor entry), then
// over (query, force component).
__global__ void __launch_bounds__(128) k_predict_finish(const double* __restrict__ G, const double* __restrict__ Erow,
                                                        const double* __restrict__ gq, const int* __restrict__ perm,
                                                        int n_atoms, int D, int DP, int S, double std, double c,
                                                        int n_splits, int64_t plane_rows, int64_t n_geo, int QPB,
                                                        double* __restrict__ E, double* __restrict__ F) {
  extern __shared__ double fd[];  // QPB * D
  const int64_t b0 = (int64_t)blockIdx.x * QPB;
  const int nq = (int)min((int64_t)QPB, n_geo - b0);
  // fixed summation order (permutation-major, then split) with four independent accumulators so
  // that the L2 round trips of the gathered loads overlap (n_splits * S terms per descriptor entry)
  const int64_t stride = plane_rows * DP;
  for (int e = threadIdx.x; e < nq * D; e += blockDim.x) {
    const int ql = e / D, d = e - ql * D;
    const int64_t b = b0 + ql;
    double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
    for (int pp = 0; pp < S; ++pp) {
      const double* gp = G + (b * S + pp) * DP + perm[pp * D + d];
      int sp = 0;
      for (; sp + 4 <= n_splits; sp += 4) {
        acc0 += gp[(int64_t)sp * stride];
        acc1 += gp[(int64_t)(sp + 1) * stride];
        acc2 += gp[(int64_t)(sp + 2) * stride];
        acc3 += gp[(int64_t)(sp + 3) * stride];
      }
      for (; sp < n_splits; ++sp) acc0 += gp[(int64_t)sp * stride];
    }
    fd[e] = (acc0 + acc1) + (acc2 + acc3);
  }
  __syncthreads();
  const int dimi = 3 * n_atoms;
  for (int e = threadIdx.x; e < nq * dimi; e += blockDim.x) {
    const int ql = e / dimi, idx = e - ql * dimi;
    const int64_t b = b0 + ql;
    const double* g = gq + b * (int64_t)D * 3;
    const double* f = fd + ql * D;
    const int k = idx / 3, cc = idx - 3 * k;
    double s = 0.0;
    for (int o = 0; o < n_atoms; ++o) {
      if (o == k) continue;
      if (o > k) {
        const int d = pair_index(o, k);
        s += g[d * 3 + cc] * f[d];
      } else {
        const int d = pair_index(k, o);
        s -= g[d * 3 + cc] * f[d];
      }
    }
    F[b * dimi + idx] = s * std;
  }
  if (E != nullptr) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int ql = warp; ql < nq; ql += (int)(blockDim.x >> 5)) {
      const int64_t b = b0 + ql;
      double s = 0.0;
      for (int t = lane; t < n_splits * S; t += 32) {
        const int sp = t / S, pp = t - sp * S;
        s += Erow[(int64_t)sp * plane_rows + b * S + pp];
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) E[b] = s * std + c;
    }
  }
}

// The same for batches of a few queries (the MD latency path: one geometry per call).  There the one-CTA-per-query form
// is a chain of S * n_splits dependent L2 round trips per thread (126 at BASELINE config 2, B = 1: ~25 us); here 1024
// threads split every descriptor entry's terms into `parts` interleaved partial sums (fixed order: bit-reproducible).
__global__ void __launch_bounds__(1024) k_predict_finish_small(const double* __restrict__ G, const double* __restrict__ Erow,
                                                               const double* __restrict__ gq, const int* __restrict__ perm,
                                                               int n_atoms, int D, int DP, int S, double std, double c,
                                                               int n_splits, int64_t plane_rows, int parts,
                                                               double* __restrict__ E, double* __restrict__ F) {
  extern __shared__ double fds[];  // parts * D partial sums, then D totals
  double* fd = fds + parts * D;
  const int64_t b = blockIdx.x;
  const int64_t stride = plane_rows * DP;
  const int n_terms = S * n_splits;
  for (int e = threadIdx.x; e < parts * D; e += blockDim.x) {
    const int part = e / D, d = e - part * D;
    double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
    int t = part;
    for (; t + 3 * parts < n_terms; t += 4 * parts) {
      const int t1 = t + parts, t2 = t + 2 * parts, t3 = t + 3 * parts;
      acc0 += G[(b * S + t % S) * DP + perm[(t % S) * D + d] + (int64_t)(t / S) * stride];
      acc1 += G[(b * S + t1 % S) * DP + perm[(t1 % S) * D + d] + (int64_t)(t1 / S) * stride];
      acc2 += G[(b * S + t2 % S) * DP + perm[(t2 % S) * D + d] + (int64_t)(t2 / S) * stride];
      acc3 += G[(b * S + t3 % S) * DP + perm[(t3 % S) * D + d] + (int64_t)(t3 / S) * stride];
    }
    for (; t < n_terms; t += parts) acc0 += G[(b * S + t % S) * DP + perm[(t % S) * D + d] + (int64_t)(t / S) * stride];
    fds[e] = (acc0 + acc1) + (acc2 + acc3);
  }
  __syncthreads();
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    double sum = 0.0;
    for (int part = 0; part < parts; ++part) sum += fds[part * D + d];
    fd[d] = sum;
  }
  __syncthreads();
  const int dimi = 3 * n_atoms;
  const double* g = gq + b * (int64_t)D * 3;
  for (int idx = threadIdx.x; idx < dimi; idx += blockDim.x) {
    const int k = idx / 3, cc = idx - 3 * k;
    double sum = 0.0;
    for (int o = 0; o < n_atoms; ++o) {
      if (o == k) continue;
      if (o > k) {
        const int d = pair_index(o, k);
        sum += g[d * 3 + cc] * fd[d];
      } else {
        const int d = pair_index(k, o);
        sum -= g[d * 3 + cc] * fd[d];
      }
    }
    F[b * dimi + idx] = sum * std;
  }
  if (E != nullptr && threadIdx.x >= blockDim.x - 32) {  // last warp
    const int lane = threadIdx.x & 31;
    double sum = 0.0;
    for (int t = lane; t < n_terms; t += 32) {
      const int sp = t / S, pp = t - sp * S;
      sum += Erow[(int64_t)sp * plane_rows + b * S + pp];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) E[b] = sum * std + c;
  }
}

// ============================================================== model maintenance kernels
__global__ void k_col_mean(const double* __restrict__ X, int M, int D, double* __restrict__ mu, int DP) {
  // one block per column
  const int d = blockIdx.x;
  __shared__ double red[256];
  double s = 0.0;
  if (d < D)
    for (int m = threadIdx.x; m < M; m += blockDim.x) s += X[(int64_t)m * D + d];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0 && d < DP) mu[d] = (d < D) ? red[0] / (double)M : 0.0;
}

// src (M, D) -> dst (Mpad, DS) zero padded, optionally centred
__global__ void k_pad_rows(const double* __restrict__ src, const double* __restrict__ mu, int M, int D, int Mpad,
                           int DS, double* __restrict__ dst) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)Mpad * DS) return;
  const int m = (int)(idx / DS), d = (int)(idx - (int64_t)m * DS);
  double v = 0.0;
  if (m < M && d < D) v = src[(int64_t)m * D + d] - (mu ? mu[d] : 0.0);
  dst[idx] = v;
}

// JA[m][d] = g_{m,d} . (alpha_{m,b} - alpha_{m,a})  (desc.py:368-385), written into the padded layout
__global__ void k_set_alphas(const double* __restrict__ R_d_desc, const double* __restrict__ alphas, int M, int D,
                             int n_atoms, int DS, double* __restrict__ JA) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)M * D) return;
  const int m = (int)(idx / D), d = (int)(idx - (int64_t)m * D);
  int a, b;
  pair_from_d(d, a, b);
  const double* v = alphas + (int64_t)m * 3 * n_atoms;
  const double* g = R_d_desc + idx * 3;
  double s = g[0] * (v[3 * b + 0] - v[3 * a + 0]);
  s += g[1] * (v[3 * b + 1] - v[3 * a + 1]);
  s += g[2] * (v[3 * b + 2] - v[3 * a + 2]);
  JA[(int64_t)m * DS + d] = s;
}

// mm[m] = |Xc_m|^2, xja[m] = Xc_m . JA_m ; one warp per row
__global__ void k_row_dots(const double* __restrict__ Xc, const double* __restrict__ JA, int Mpad, int DS,
                           double* __restrict__ mm, double* __restrict__ xja) {
  const int m = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (m >= Mpad) return;
  double s1 = 0.0, s2 = 0.0;
  for (int d = lane; d < DS; d += 32) {
    const double x = Xc[(int64_t)m * DS + d];
    s1 = fma(x, x, s1);
    s2 = fma(x, JA[(int64_t)m * DS + d], s2);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  if (lane == 0) {
    if (mm) mm[m] = s1;
    xja[m] = s2;
  }
}

__global__ void k_unpad_rows(const double* __restrict__ src, int M, int D, int DS, double* __restrict__ dst) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)M * D) return;
  const int m = (int)(idx / D), d = (int)(idx - (int64_t)m * D);
  dst[idx] = src[(int64_t)m * DS + d];
}

}  // namespace sgdml

using namespace sgdml;

// ============================================================== model object
struct sgdml_b200_model {
  int N = 0, D = 0, M = 0, S = 0;
  int DP = 0, DS = 0, BM = 0, BQ = 0, Mpad = 0, cfg = -1;
  int device = 0;
  bool large = false;                    // D > 256: GEMM-composed path
  double *XcT = nullptr, *JAT = nullptr;  // (DP, Mpad) transposed copies for the second contraction
  double sig = 0, std = 1, c = 0;
  double *X = nullptr;    // (M, D) raw descriptors (training-point queries)
  double *Xc = nullptr, *JA = nullptr, *mm = nullptr, *xja = nullptr, *mu = nullptr;
  // large descriptors: the four contractions on the tcgen05 tensor cores through int8 slices (csrc/ozaki.cu) when
  // oz_s >= 2; the slices of the model matrices are kept (those of JA / JA^T are refreshed by set_alphas)
  int oz_s = 0;
  OzOperand ozXc, ozJA, ozXcT, ozJAT;
  double* ae = nullptr;                  // (Mpad) alphas_E, zeros unless use_ae
  int use_ae = 0;
  Lattice lat = {0, {0}, {0}};           // periodic cell of the query descriptors (predict.py:332-334)
  int *perm = nullptr, *pinv = nullptr;  // (S, D)
  double* R_d_desc = nullptr;            // (M, D, 3), optional
  // two workspace slots (slot 1 and the side streams are only used by the host-I/O pipeline)
  struct WS {
    int64_t geo = 0;
    double *xq = nullptr, *gq = nullptr, *G = nullptr, *Erow = nullptr, *R = nullptr, *E = nullptr, *F = nullptr,
           *Qg = nullptr, *qq = nullptr, *S1 = nullptr, *S2 = nullptr, *csum = nullptr;
    OzOperand ozQ, ozC1, ozC2;  // slices of the per-batch operands (int8 path of large descriptors)
  } ws[2];
  cudaStream_t pipe_stream[2] = {nullptr, nullptr};
  cudaEvent_t pipe_event[3] = {nullptr, nullptr, nullptr};
  // MD latency path: the launch sequence of a small host-buffer batch, captured once per batch size into a CUDA graph
  struct GraphSlot {
    int64_t n_geo = 0;
    int with_E = 0;
    int n_kernels = 0;
    uint64_t generation = 0;
    cudaGraphExec_t exec = nullptr;
    double *hR = nullptr, *hF = nullptr, *hE = nullptr;  // pinned staging
  } graphs[4];
  int graph_next = 0;
  uint64_t generation = 1;  // bumped whenever something a captured graph has baked in changes (workspace, cell, alphas_E)
  cudaStream_t graph_stream = nullptr;
  cudaEvent_t graph_event = nullptr;
};

namespace {

// tile configurations: <DP, BQ, BM, W1Q, W1M, W1K, W2Q, W2D>
// D <= 40: two co-resident CTAs per SM so that one CTA's transform / barriers / prologue overlap
// the other's DMMA phases (the sweep over M is only a handful of tiles at ethanol size)
using Cfg40 = PCfg<40, 64, 32, 4, 2, 1, 4, 1, 2, 2>;
using Cfg72 = PCfg<72, 64, 32, 4, 2, 1, 8, 1>;
using Cfg112 = PCfg<112, 64, 16, 4, 1, 2, 4, 2>;
using Cfg160 = PCfg<160, 32, 16, 2, 1, 4, 2, 4>;
using Cfg224 = PCfg<224, 32, 16, 2, 1, 4, 2, 4>;
using Cfg256 = PCfg<256, 32, 8, 2, 1, 4, 2, 4>;
// variant 2: the same tiles without the split over k -- every warp owns whole S1 / S2 fragments, the Matern transform
// runs on the accumulator registers and one of the three barriers per tile (and the partial-sum round trip through
// shared memory) goes away; the price is three operand loads per two DMMAs in GEMM1
using Cfg112f = PCfg<112, 64, 16, 4, 2, 1, 4, 2>;
using Cfg160f = PCfg<160, 32, 16, 4, 2, 1, 2, 4>;
using Cfg224f = PCfg<224, 32, 16, 4, 2, 1, 2, 4>;
// variant 3: variant 2 with one barrier per tile (OB), for every descriptor size up to 224
using Cfg40o = PCfg<40, 64, 32, 4, 2, 1, 4, 1, 2, 2, 1>;
using Cfg72o = PCfg<72, 64, 32, 4, 2, 1, 8, 1, 1, 1, 1>;
using Cfg112o = PCfg<112, 64, 16, 4, 2, 1, 4, 2, 1, 1, 1>;
using Cfg160o = PCfg<160, 32, 16, 4, 2, 1, 2, 4, 1, 1, 1>;
using Cfg224o = PCfg<224, 32, 16, 4, 2, 1, 2, 4, 1, 1, 1>;
// variant 5 (DP = 40 only): the one-barrier form on 16-point tiles, which keeps two CTAs per SM (88 KB)
using Cfg40o16 = PCfg<40, 64, 16, 4, 2, 1, 4, 1, 2, 2, 1>;

struct CfgInfo {
  int DP, BQ, BM;
};
const CfgInfo kCfgs[] = {{40, 64, 32}, {72, 64, 32}, {112, 64, 16}, {160, 32, 16}, {224, 32, 16}, {256, 32, 8}};
const int kNumCfgs = 6;

template <class C>
int launch_main_pp_t(const PredictArgs& a, int n_splits, cudaStream_t s) {
  static bool configured[64] = {false};
  int dev = 0;
  SG_CUDA(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && !configured[dev]) {
    SG_CUDA(cudaFuncSetAttribute(k_predict_main_pp<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PPCfg<C>::SMEM_BYTES));
    configured[dev] = true;
  }
  const int64_t grid = (a.n_rows + C::BQ - 1) / C::BQ;
  k_predict_main_pp<C><<<dim3((unsigned)grid, (unsigned)n_splits), C::NT, PPCfg<C>::SMEM_BYTES, s>>>(a);
  SG_CUDA(cudaGetLastError());
  return 0;
}

template <class C>
int launch_main_t(const PredictArgs& a, int n_splits, cudaStream_t s) {
  static bool configured[64] = {false};
  int dev = 0;
  SG_CUDA(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && !configured[dev]) {
    SG_CUDA(cudaFuncSetAttribute(k_predict_main<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM_BYTES));
    configured[dev] = true;
  }
  const int64_t grid = (a.n_rows + C::BQ - 1) / C::BQ;
  PredictArgs b = a;
  if (a.bm > C::BM) b.tiles_per_split = a.tiles_per_split * (a.bm / C::BM);  // (a.bm is a multiple of C::BM)
  k_predict_main<C><<<dim3((unsigned)grid, (unsigned)n_splits), C::NT, C::SMEM_BYTES, s>>>(b);
  SG_CUDA(cudaGetLastError());
  return 0;
}

int g_predict_variant = 0;  // see sgdml_b200_set_predict_variant (include/sgdml_b200.h)

int launch_main(int cfg, const PredictArgs& a, int n_splits, cudaStream_t s) {
  if (g_predict_variant == 1) {
    switch (cfg) {
      case 2: return launch_main_pp_t<Cfg112>(a, n_splits, s);
      case 3: return launch_main_pp_t<Cfg160>(a, n_splits, s);
      case 4: return launch_main_pp_t<Cfg224>(a, n_splits, s);
      case 5: return launch_main_pp_t<Cfg256>(a, n_splits, s);
    }
  }
  if (g_predict_variant == 2) {
    switch (cfg) {
      case 2: return launch_main_t<Cfg112f>(a, n_splits, s);
      case 3: return launch_main_t<Cfg160f>(a, n_splits, s);
      case 4: return launch_main_t<Cfg224f>(a, n_splits, s);
    }
  }
  if (g_predict_variant == 3) {
    switch (cfg) {
      case 0: return launch_main_t<Cfg40o>(a, n_splits, s);
      case 1: return launch_main_t<Cfg72o>(a, n_splits, s);
      case 2: return launch_main_t<Cfg112o>(a, n_splits, s);
      case 3: return launch_main_t<Cfg160o>(a, n_splits, s);
      case 4: return launch_main_t<Cfg224o>(a, n_splits, s);
    }
  }
  if (g_predict_variant == 5 && cfg == 0) return launch_main_t<Cfg40o16>(a, n_splits, s);
  if (g_predict_variant == 0) {
    // default: the measured-fastest kernel per size (tools/predict_variants.py, 65536 queries, M = 1000, S = 6, ms per
    // call round-1 kernel -> one-barrier kernel): DP = 72: 9.09 -> 8.89, 112: 13.98 -> 12.73, 160: 20.07 -> 18.12,
    // 224 (BASELINE config 2): 25.81 -> 24.01; DP = 40 (config 1) stays on the round-1 kernel (1.31 vs 1.51 ms: the
    // doubled C1 / C2 buffers cost it its second CTA per SM)
    switch (cfg) {
      case 1: return launch_main_t<Cfg72o>(a, n_splits, s);
      case 2: return launch_main_t<Cfg112o>(a, n_splits, s);
      case 3: return launch_main_t<Cfg160o>(a, n_splits, s);
      case 4: return launch_main_t<Cfg224o>(a, n_splits, s);
    }
  }
  switch (cfg) {  // (variant 4: the round-1 kernels for every size)
    case 0: return launch_main_t<Cfg40>(a, n_splits, s);
    case 1: return launch_main_t<Cfg72>(a, n_splits, s);
    case 2: return launch_main_t<Cfg112>(a, n_splits, s);
    case 3: return launch_main_t<Cfg160>(a, n_splits, s);
    case 4: return launch_main_t<Cfg224>(a, n_splits, s);
    case 5: return launch_main_t<Cfg256>(a, n_splits, s);
  }
  return fail_arg("no predictor tile configuration for this descriptor size");
}

int64_t chunk_geos(const sgdml_b200_model* m);

void free_oz(OzOperand& o) {
  cached_free(o.units);
  cached_free(o.exps);
  o = OzOperand();
}

int alloc_oz(OzOperand& o, int64_t rows, int64_t k, int S) {
  if (o.units != nullptr) cudaDeviceSynchronize();  // (blocks go back to the cache: nothing may still use them)
  free_oz(o);
  SG_CUDA(cached_malloc(&o.units, ozaki_units_bytes(rows, k, S)));
  SG_CUDA(cached_malloc(&o.exps, ozaki_exps_bytes(rows)));
  return 0;
}

void free_ws(sgdml_b200_model* m) {
  cudaDeviceSynchronize();  // the blocks go back to the cache (no implicit synchronisation as in cudaFree)
  for (auto& w : m->ws) {
    free_oz(w.ozQ);
    free_oz(w.ozC1);
    free_oz(w.ozC2);
    cached_free(w.xq);
    cached_free(w.gq);
    cached_free(w.G);
    cached_free(w.Erow);
    cached_free(w.R);
    cached_free(w.E);
    cached_free(w.F);
    cached_free(w.Qg);
    cached_free(w.qq);
    cached_free(w.S1);
    cached_free(w.S2);
    cached_free(w.csum);
    w = sgdml_b200_model::WS();
  }
}

int ensure_ws(sgdml_b200_model* m, int slot, int64_t n_geo) {
  sgdml_b200_model::WS& w = m->ws[slot];
  if (!m->large) {  // room for the per-split output planes of small batches (<= ~300 CTAs x BQ rows)
    const int64_t min_geo = (int64_t)(2 * 148 + 8) * m->BQ / m->S + 1;
    n_geo = std::max<int64_t>(n_geo, std::min<int64_t>(min_geo, chunk_geos(m)));
  }
  if (n_geo <= w.geo) return 0;
  ++m->generation;  // captured graphs hold the old workspace pointers
  if (w.geo > 0) SG_CUDA(cudaDeviceSynchronize());  // earlier batches may still run on the old workspace
  free_oz(w.ozQ);
  free_oz(w.ozC1);
  free_oz(w.ozC2);
  cached_free(w.xq);
  cached_free(w.gq);
  cached_free(w.G);
  cached_free(w.Erow);
  cached_free(w.R);
  cached_free(w.E);
  cached_free(w.F);
  cached_free(w.Qg);
  cached_free(w.qq);
  cached_free(w.S1);
  cached_free(w.S2);
  cached_free(w.csum);
  w = sgdml_b200_model::WS();
  SG_CUDA(cached_malloc(&w.xq, sizeof(double) * n_geo * m->D));
  SG_CUDA(cached_malloc(&w.gq, sizeof(double) * n_geo * m->D * 3));
  {
    // padded to whole row tiles: the per-split output planes of small batches are laid out with that stride
    const int64_t rows_cap = (n_geo * m->S + m->BQ - 1) / m->BQ * m->BQ;
    SG_CUDA(cached_malloc(&w.G, sizeof(double) * rows_cap * m->DP));
    SG_CUDA(cached_malloc(&w.Erow, sizeof(double) * rows_cap));
  }
  SG_CUDA(cached_malloc(&w.R, sizeof(double) * n_geo * 3 * m->N));
  SG_CUDA(cached_malloc(&w.E, sizeof(double) * n_geo));
  SG_CUDA(cached_malloc(&w.F, sizeof(double) * n_geo * 3 * m->N));
  {
    const int64_t rows_pad = (n_geo * m->S + m->BQ - 1) / m->BQ * m->BQ;
    SG_CUDA(cached_malloc(&w.Qg, sizeof(double) * rows_pad * m->DS));
    SG_CUDA(cached_malloc(&w.qq, sizeof(double) * rows_pad));
    if (m->large) {
      SG_CUDA(cached_malloc(&w.S1, sizeof(double) * rows_pad * m->Mpad));
      SG_CUDA(cached_malloc(&w.S2, sizeof(double) * rows_pad * m->Mpad));
      SG_CUDA(cached_malloc(&w.csum, sizeof(double) * rows_pad));
      if (m->oz_s >= 2) {
        SG_TRY(alloc_oz(w.ozQ, rows_pad, m->DS, m->oz_s));
        SG_TRY(alloc_oz(w.ozC1, rows_pad, m->Mpad, m->oz_s));
        SG_TRY(alloc_oz(w.ozC2, rows_pad, m->Mpad, m->oz_s));
      }
    }
  }
  w.geo = n_geo;
  return 0;
}

int ensure_pipe(sgdml_b200_model* m) {
  if (m->pipe_stream[0] != nullptr) return 0;
  for (int i = 0; i < 2; ++i) SG_CUDA(cudaStreamCreateWithFlags(&m->pipe_stream[i], cudaStreamNonBlocking));
  for (int i = 0; i < 3; ++i) SG_CUDA(cudaEventCreateWithFlags(&m->pipe_event[i], cudaEventDisableTiming));
  return 0;
}

// queries per chunk: bounds the G workspace (rows * DP * 8 bytes) to ~256 MB
int64_t chunk_geos(const sgdml_b200_model* m) {
  int64_t rows = (int64_t)(256ll << 20) / ((int64_t)m->DP * 8);
  if (m->large) rows = std::min<int64_t>((int64_t)(2048ll << 20) / ((int64_t)m->DP * 8), (int64_t)(2048ll << 20) / ((int64_t)m->Mpad * 8));
  int64_t g = rows / m->S;
  if (g < 1) g = 1;
  if (g > 65536) g = 65536;
  return g;
}

// Runs the predictor on n_geo queries whose descriptors (xq, gq) are on the device.
constexpr int64_t GRAPH_MAX_GEO = 16;  // batches up to this size with host buffers replay a captured graph
// xq == nullptr: the query rows (w.Qg, w.qq) are already in place (k_desc_query_rows)
// n_splits_out (optional): number of per-split G / Erow planes left in the workspace (stride: rows rounded up to BQ);
// fp64: the large-descriptor contractions in FP64 DMMA even when the model uses int8 slices
int run_queries(sgdml_b200_model* m, int slot, const double* xq, const double* gq, int64_t n_geo, double std,
                double c, double* E_dev, double* F_dev, cudaStream_t s, int* n_splits_out = nullptr,
                bool fp64 = false) {
  sgdml_b200_model::WS& w = m->ws[slot];
  const int64_t n_rows = n_geo * m->S;
  const int64_t n_rows_pad = (n_rows + m->BQ - 1) / m->BQ * m->BQ;
  int n_splits = 1;
  if (xq != nullptr) {
    ProfScope ps(KID_PREDICT_AUX, s);
    k_query_rows<<<(unsigned)((n_rows_pad + 7) / 8), 256, 0, s>>>(xq, m->pinv, m->mu, m->D, m->DS, m->S, n_rows,
                                                                 n_rows_pad, w.Qg, w.qq);
    SG_CUDA(cudaGetLastError());
    count_launch(KID_PREDICT_AUX);
  }
  if (m->large) {
    ProfScope ps(KID_PREDICT_MAIN, s);
    MaternK mk;
    mk.sig = m->sig;
    mk.sig_inv = 1.0 / m->sig;
    mk.k_base = 5.0 / (3.0 * m->sig * m->sig * m->sig);
    mk.k_c1 = mk.k_base * 5.0 / m->sig;
    GemmArgs g;
    g.alpha = 1.0;
    g.beta = 0.0;
    g.mode = 0;
    g.tri = 0;
    g.abort_flag = nullptr;
    // The four contractions on the tcgen05 tensor cores through exact int8 slice products (csrc/ozaki.cu): the
    // slices of the model matrices are kept with the model, those of Q, C1, C2 are cut per batch; everything is
    // stream-ordered (this path runs once per CG iteration inside sgdml_b200_pcg).  Slice count: m->oz_s
    // (tools/ozaki_study.py predict: forces 8.8e-9 / 6.5e-11 / 5.4e-13 vs FP64 for 4 / 5 / 6 slices).
    if (m->oz_s >= 2 && !fp64) {
      const int S = m->oz_s;
      SG_TRY(ozaki_split(w.Qg, n_rows, m->DS, m->DS, S, w.ozQ.units, w.ozQ.exps, &w.ozQ, s));
      SG_TRY(ozaki_gemm(w.ozQ, m->ozXc, n_rows, m->Mpad, 1.0, 1, w.S1, m->Mpad, S, s));
      SG_TRY(ozaki_gemm(w.ozQ, m->ozJA, n_rows, m->Mpad, 1.0, 1, w.S2, m->Mpad, S, s));
      k_transform_rows<<<(unsigned)((n_rows + 7) / 8), 256, 0, s>>>(w.S1, w.S2, m->Mpad, w.qq, m->mm, m->xja, m->use_ae ? m->ae : nullptr, m->M,
                                                                     m->Mpad, n_rows, mk, w.csum, w.Erow);
      SG_CUDA(cudaGetLastError());
      SG_TRY(ozaki_split(w.S1, n_rows, m->Mpad, m->Mpad, S, w.ozC1.units, w.ozC1.exps, &w.ozC1, s));
      SG_TRY(ozaki_split(w.S2, n_rows, m->Mpad, m->Mpad, S, w.ozC2.units, w.ozC2.exps, &w.ozC2, s));
      SG_TRY(ozaki_gemm(w.ozC1, m->ozXcT, n_rows, m->DP, 1.0, 1, w.G, m->DP, S, s));
      SG_TRY(ozaki_gemm(w.ozC2, m->ozJAT, n_rows, m->DP, 1.0, 0, w.G, m->DP, S, s));
    } else {
    // S1 = Q Xc^T, S2 = Q JA^T   (rows x Mpad, contraction over the padded descriptor)
    g.m = n_rows;
    g.n = m->Mpad;
    g.k = m->DS;
    g.A = w.Qg;
    g.lda = m->DS;
    g.ldb = m->DS;
    g.ldc = m->Mpad;
    g.B = m->Xc;
    g.C = w.S1;
    SG_TRY(launch_gemm(g, s));
    g.B = m->JA;
    g.C = w.S2;
    SG_TRY(launch_gemm(g, s));
    k_transform_rows<<<(unsigned)((n_rows + 7) / 8), 256, 0, s>>>(w.S1, w.S2, m->Mpad, w.qq, m->mm, m->xja, m->use_ae ? m->ae : nullptr, m->M,
                                                                   m->Mpad, n_rows, mk, w.csum, w.Erow);
    SG_CUDA(cudaGetLastError());
    // acc = C1 XcT^T + C2 JAT^T   (rows x DP, contraction over the training points)
    g.n = m->DP;
    g.k = m->Mpad;
    g.lda = m->Mpad;
    g.ldb = m->Mpad;
    g.ldc = m->DP;
    g.A = w.S1;
    g.B = m->XcT;
    g.C = w.G;
    SG_TRY(launch_gemm(g, s));
    g.mode = 1;
    g.A = w.S2;
    g.B = m->JAT;
    SG_TRY(launch_gemm(g, s));
    }
    k_combine_rows<<<(unsigned)((n_rows * m->DP + 255) / 256), 256, 0, s>>>(w.Qg, m->DS, w.csum, w.G, m->DP, n_rows);
    SG_CUDA(cudaGetLastError());
    count_launch(KID_PREDICT_MAIN, 2);
  } else {
    PredictArgs a;
    a.Xc = m->Xc;
    a.JA = m->JA;
    a.mm = m->mm;
    a.xja = m->xja;
    a.ae = m->ae;
    a.use_ae = m->use_ae;
    a.D = m->D;
    a.M = m->M;
    a.S = m->S;
    a.Mpad = m->Mpad;
    a.sig = m->sig;
    a.Qg = w.Qg;
    a.qqg = w.qq;
    a.n_rows = n_rows;
    a.n_rows_pad = n_rows_pad;
    a.bm = m->BM;
    a.G = w.G;
    a.Erow = w.Erow;
    // small batches: split the sweep over the training points across CTAs so that the grid fills the
    // GPU (partial G / E planes are summed by the finishing kernel); bounded by the workspace capacity
    {
      const int n_tiles = m->Mpad / m->BM;
      const int64_t q_tiles = n_rows_pad / m->BQ;
      const int64_t target = 2 * (int64_t)num_sms();
      int64_t sp = (target + q_tiles - 1) / q_tiles;
      const int64_t cap_rows = (w.geo * m->S + m->BQ - 1) / m->BQ * m->BQ;
      sp = std::min<int64_t>(sp, cap_rows / n_rows_pad);
      sp = std::min<int64_t>(sp, 2 * (int64_t)std::ceil(std::sqrt(2.0 * n_tiles)));  // finishing cost grows with splits
      sp = std::max<int64_t>(1, std::min<int64_t>(sp, n_tiles));
      a.tiles_per_split = (int)((n_tiles + sp - 1) / sp);
      n_splits = (n_tiles + a.tiles_per_split - 1) / a.tiles_per_split;
    }
    ProfScope ps(KID_PREDICT_MAIN, s);
    SG_TRY(launch_main(m->cfg, a, n_splits, s));
    count_launch(KID_PREDICT_MAIN);
  }
  {
    ProfScope ps(KID_PREDICT_AUX, s);
    const int QPB = std::max(1, 128 / m->D);  // small molecules: several queries per CTA
    const size_t fd_bytes = sizeof(double) * (size_t)m->D * QPB;
    if (fd_bytes > 48 * 1024) {  // molecules above 111 atoms: opt in to more than the default dynamic shared memory
      if (fd_bytes > 200 * 1024) {
        set_last_error("sgdml_b200_predict: descriptor too long for the finishing kernel (n_atoms <= ~225 supported)");
        return SGDML_B200_ERR_UNSUPPORTED;
      }
      SG_CUDA(cudaFuncSetAttribute(k_predict_finish, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fd_bytes));
    }
    const int parts = std::max(1, std::min(8, 1024 / m->D));
    const size_t fds_bytes = sizeof(double) * (size_t)m->D * (parts + 1);
    if (n_geo <= GRAPH_MAX_GEO && n_splits > 1 && parts > 1 && fds_bytes <= 48 * 1024) {
      // a few queries, the sweep over the training points split across CTAs: the latency form
      k_predict_finish_small<<<(unsigned)n_geo, 1024, fds_bytes, s>>>(w.G, w.Erow, gq, m->perm, m->N, m->D, m->DP, m->S, std, c,
                                                                     n_splits, n_rows_pad, parts, E_dev, F_dev);
    } else {
      k_predict_finish<<<(unsigned)((n_geo + QPB - 1) / QPB), 128, fd_bytes, s>>>(w.G, w.Erow, gq, m->perm, m->N, m->D,
                                                                                 m->DP, m->S, std, c, n_splits,
                                                                                 n_rows_pad, n_geo, QPB, E_dev, F_dev);
    }
    SG_CUDA(cudaGetLastError());
    count_launch(KID_PREDICT_AUX);
  }
  if (n_splits_out != nullptr) *n_splits_out = n_splits;
  return 0;
}

int refresh_transposes(sgdml_b200_model* m, bool with_x, cudaStream_t s) {
  dim3 grid((unsigned)((m->DP + 31) / 32), (unsigned)((m->Mpad + 31) / 32));
  if (with_x) k_transpose_pad<<<grid, dim3(32, 8), 0, s>>>(m->Xc, m->Mpad, m->DP, m->DS, m->XcT, m->Mpad);
  k_transpose_pad<<<grid, dim3(32, 8), 0, s>>>(m->JA, m->Mpad, m->DP, m->DS, m->JAT, m->Mpad);
  SG_CUDA(cudaGetLastError());
  count_launch(KID_PREDICT_AUX, with_x ? 2 : 1);
  return 0;
}

// (re)cuts the model matrices into int8 slices: Xc / Xc^T once, JA / JA^T after every set_alphas
int refresh_oz_model(sgdml_b200_model* m, bool with_x, cudaStream_t s) {
  if (m->oz_s < 2) return 0;
  const int S = m->oz_s;
  if (with_x) {
    SG_TRY(alloc_oz(m->ozXc, m->Mpad, m->DS, S));
    SG_TRY(alloc_oz(m->ozJA, m->Mpad, m->DS, S));
    SG_TRY(alloc_oz(m->ozXcT, m->DP, m->Mpad, S));
    SG_TRY(alloc_oz(m->ozJAT, m->DP, m->Mpad, S));
    SG_TRY(ozaki_split(m->Xc, m->Mpad, m->DS, m->DS, S, m->ozXc.units, m->ozXc.exps, &m->ozXc, s));
    SG_TRY(ozaki_split(m->XcT, m->DP, m->Mpad, m->Mpad, S, m->ozXcT.units, m->ozXcT.exps, &m->ozXcT, s));
  }
  SG_TRY(ozaki_split(m->JA, m->Mpad, m->DS, m->DS, S, m->ozJA.units, m->ozJA.exps, &m->ozJA, s));
  SG_TRY(ozaki_split(m->JAT, m->DP, m->Mpad, m->Mpad, S, m->ozJAT.units, m->ozJAT.exps, &m->ozJAT, s));
  return 0;
}

int refresh_row_dots(sgdml_b200_model* m, bool with_mm, cudaStream_t s) {
  k_row_dots<<<ceil_div(m->Mpad, 8), 256, 0, s>>>(m->Xc, m->JA, m->Mpad, m->DS, with_mm ? m->mm : nullptr, m->xja);
  SG_CUDA(cudaGetLastError());
  count_launch(KID_PREDICT_AUX);
  return 0;
}

}  // namespace

extern "C" {

int sgdml_b200_model_create(sgdml_b200_model** out, int64_t n_atoms, int64_t n_train, int64_t n_perms,
                            const double* R_desc, const double* R_d_desc_alpha, const int64_t* tril_perms_lin,
                            double sig, double std, double c) {
  SG_TRY(require_device());
  SG_ARG(out != nullptr && R_desc != nullptr && R_d_desc_alpha != nullptr && tril_perms_lin != nullptr);
  SG_ARG(n_atoms >= 2 && n_train >= 1 && n_perms >= 1 && sig > 0);
  const int64_t D = n_atoms * (n_atoms - 1) / 2;
  int cfg = -1;
  for (int i = 0; i < kNumCfgs; ++i)
    if (D <= kCfgs[i].DP) {
      cfg = i;
      break;
    }
  sgdml_b200_model* m = new sgdml_b200_model();
  m->N = (int)n_atoms;
  m->D = (int)D;
  m->M = (int)n_train;
  m->S = (int)n_perms;
  m->cfg = cfg;
  if (cfg >= 0) {
    m->DP = kCfgs[cfg].DP;
    m->BQ = kCfgs[cfg].BQ;
    m->BM = kCfgs[cfg].BM;
  } else {
    // D > 256 (N > 23 atoms): GEMM-composed path, any descriptor size
    m->large = true;
    m->DP = (int)((D + 7) / 8 * 8);
    m->BQ = 8;
    m->BM = 8;
  }
  m->DS = m->DP + 4;
  m->Mpad = (int)((n_train + m->BM - 1) / m->BM * m->BM);
  m->sig = sig;
  m->std = std;
  m->c = c;
  cudaGetDevice(&m->device);

  // integer tables on the host (bit-exact), then to the device
  std::vector<int64_t> lin((size_t)(n_perms * D));
  if (is_device_ptr(tril_perms_lin)) {
    cudaError_t e = cudaMemcpy(lin.data(), tril_perms_lin, sizeof(int64_t) * lin.size(), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) {
      delete m;
      return fail_cuda(e, "copy tril_perms_lin", __FILE__, __LINE__);
    }
  } else {
    std::copy(tril_perms_lin, tril_perms_lin + lin.size(), lin.begin());
  }
  std::vector<int> perm((size_t)(n_perms * D)), pinv((size_t)(n_perms * D), -1);
  for (int64_t pp = 0; pp < n_perms; ++pp)
    for (int64_t d = 0; d < D; ++d) {
      const int64_t e = lin[(size_t)(d * n_perms + pp)] - pp * D;  // train.py:903-904
      if (e < 0 || e >= D || pinv[(size_t)(pp * D + e)] != -1) {
        delete m;
        return fail_arg("tril_perms_lin must encode S permutations of 0..D-1");
      }
      perm[(size_t)(pp * D + d)] = (int)e;
      pinv[(size_t)(pp * D + e)] = (int)d;
    }

  int rc = 0;
  auto body = [&]() -> int {
    cudaStream_t s = 0;
    SG_CUDA(cached_malloc(&m->perm, sizeof(int) * perm.size()));
    SG_CUDA(cached_malloc(&m->pinv, sizeof(int) * pinv.size()));
    SG_CUDA(cudaMemcpy(m->perm, perm.data(), sizeof(int) * perm.size(), cudaMemcpyHostToDevice));
    SG_CUDA(cudaMemcpy(m->pinv, pinv.data(), sizeof(int) * pinv.size(), cudaMemcpyHostToDevice));
    SG_CUDA(cached_malloc(&m->X, sizeof(double) * n_train * D));
    SG_CUDA(cached_malloc(&m->Xc, sizeof(double) * m->Mpad * m->DS));
    SG_CUDA(cached_malloc(&m->JA, sizeof(double) * m->Mpad * m->DS));
    SG_CUDA(cached_malloc(&m->mm, sizeof(double) * m->Mpad));
    SG_CUDA(cached_malloc(&m->xja, sizeof(double) * m->Mpad));
    SG_CUDA(cached_malloc(&m->ae, sizeof(double) * m->Mpad));
    SG_CUDA(cudaMemset(m->ae, 0, sizeof(double) * m->Mpad));
    SG_CUDA(cached_malloc(&m->mu, sizeof(double) * m->DS));
    SG_CUDA(cudaMemset(m->mu, 0, sizeof(double) * m->DS));
    Staged sJA;
    SG_CUDA(cudaMemcpy(m->X, R_desc, sizeof(double) * n_train * D, cudaMemcpyDefault));
    SG_TRY(sJA.init(R_d_desc_alpha, sizeof(double) * n_train * D, true, s));
    k_col_mean<<<m->DP, 256, 0, s>>>(m->X, m->M, m->D, m->mu, m->DP);
    SG_CUDA(cudaGetLastError());
    const int64_t tot = (int64_t)m->Mpad * m->DS;
    k_pad_rows<<<ceil_div(tot, 256), 256, 0, s>>>(m->X, m->mu, m->M, m->D, m->Mpad, m->DS, m->Xc);
    SG_CUDA(cudaGetLastError());
    k_pad_rows<<<ceil_div(tot, 256), 256, 0, s>>>((const double*)sJA.dev(), nullptr, m->M, m->D, m->Mpad, m->DS,
                                                  m->JA);
    SG_CUDA(cudaGetLastError());
    SG_TRY(refresh_row_dots(m, true, s));
    if (m->large) {
      SG_CUDA(cached_malloc(&m->XcT, sizeof(double) * (size_t)m->DP * m->Mpad));
      SG_CUDA(cached_malloc(&m->JAT, sizeof(double) * (size_t)m->DP * m->Mpad));
      SG_TRY(refresh_transposes(m, true, s));
      const char* ozp = getenv("SGDML_B200_OZAKI_PREDICT_SLICES");
      const int oz_s = (ozp != nullptr) ? std::max(0, std::min(7, atoi(ozp))) : 0;
      if (oz_s >= 2 && m->DS <= (1 << 14) && m->Mpad <= (1 << 14)) m->oz_s = oz_s;
      SG_TRY(refresh_oz_model(m, true, s));
    }
    SG_CUDA(cudaStreamSynchronize(s));
    return 0;
  };
  rc = body();
  if (rc != 0) {
    sgdml_b200_model_destroy(m);
    return rc;
  }
  *out = m;
  return 0;
}

namespace {

// SGDML_B200_GRAPH=0 switches the CUDA-graph replay of small host-buffer batches off (measured on B200, B = 1,
// NumPy in/out: 54 vs 65 us per call at BASELINE config 1, 92 vs 105 us at config 2)
bool g_graph_enabled() {
  const char* e = getenv("SGDML_B200_GRAPH");
  return e != nullptr ? (e[0] == '1') : true;
}
bool g_graph_zero_copy() {
  const char* e = getenv("SGDML_B200_GRAPH_ZEROCOPY");
  return e != nullptr ? (e[0] == '1') : true;
}

void free_graph_slot(sgdml_b200_model::GraphSlot& g) {
  if (g.exec) cudaGraphExecDestroy(g.exec);
  cudaFreeHost(g.hR);
  cudaFreeHost(g.hF);
  cudaFreeHost(g.hE);
  g = sgdml_b200_model::GraphSlot();
}

// Small host-buffer batch (molecular dynamics: one geometry per call, ase_calc.py:98-110): pinned staging buffers and
// the whole launch sequence (H2D copy, descriptor kernel, query rows, main kernel, finishing kernel, D2H copies)
// replayed from a CUDA graph -- one launch call instead of seven.
int predict_graph(sgdml_b200_model* m, const double* R, int64_t n_geo, double* E, double* F, cudaStream_t s) {
  const int dimi = 3 * m->N;
  const int with_E = E != nullptr ? 1 : 0;
  SG_TRY(ensure_ws(m, 0, n_geo));
  if (m->graph_stream == nullptr) {
    SG_CUDA(cudaStreamCreateWithFlags(&m->graph_stream, cudaStreamNonBlocking));
    SG_CUDA(cudaEventCreateWithFlags(&m->graph_event, cudaEventDisableTiming));
  }
  cudaStream_t gs = m->graph_stream;
  sgdml_b200_model::WS& w = m->ws[0];
  sgdml_b200_model::GraphSlot* g = nullptr;
  for (auto& c : m->graphs)
    if (c.exec != nullptr && c.n_geo == n_geo && c.with_E == with_E && c.generation == m->generation) g = &c;
  // Three kernel nodes and no copy nodes: the first kernel reads the geometries straight from the pinned staging
  // buffer (unified addressing) and builds descriptors + query rows, the finishing kernel stores E and F straight
  // into pinned host memory.  SGDML_B200_GRAPH_ZEROCOPY=0: the earlier form (H2D copy, descriptor kernel, query-row
  // kernel, ..., two D2H copies).
  const size_t dq_bytes = sizeof(double) * (size_t)(dimi + m->D);
  const bool zero_copy = g_graph_zero_copy() && dq_bytes <= 200 * 1024;
  auto enqueue = [&](sgdml_b200_model::GraphSlot* q) -> int {
    if (zero_copy) {
      const int64_t n_rows = n_geo * m->S;
      const int64_t n_rows_pad = (n_rows + m->BQ - 1) / m->BQ * m->BQ;
      if (dq_bytes > 48 * 1024)
        SG_CUDA(cudaFuncSetAttribute(k_desc_query_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dq_bytes));
      k_desc_query_rows<<<(unsigned)n_geo, 256, dq_bytes, gs>>>(q->hR, m->N, m->pinv, m->mu, m->D, m->DS, m->S, n_rows,
                                                               n_rows_pad, w.gq, w.Qg, w.qq, m->lat);
      SG_CUDA(cudaGetLastError());
      count_launch(KID_PREDICT_AUX);
      SG_TRY(run_queries(m, 0, nullptr, w.gq, n_geo, m->std, m->c, with_E ? q->hE : nullptr, q->hF, gs));
      return 0;
    }
    SG_CUDA(cudaMemcpyAsync(w.R, q->hR, sizeof(double) * n_geo * dimi, cudaMemcpyHostToDevice, gs));
    SG_TRY(launch_desc_from_R(w.R, n_geo, m->N, w.xq, w.gq, gs, &m->lat));
    SG_TRY(run_queries(m, 0, w.xq, w.gq, n_geo, m->std, m->c, with_E ? w.E : nullptr, w.F, gs));
    SG_CUDA(cudaMemcpyAsync(q->hF, w.F, sizeof(double) * n_geo * dimi, cudaMemcpyDeviceToHost, gs));
    if (with_E) SG_CUDA(cudaMemcpyAsync(q->hE, w.E, sizeof(double) * n_geo, cudaMemcpyDeviceToHost, gs));
    return 0;
  };
  if (g == nullptr) {
    // capture happens on a private stream (the caller's may be the legacy stream, which cannot be captured); work
    // queued on the caller's stream (set_alphas, ...) comes first
    SG_CUDA(cudaEventRecord(m->graph_event, s));
    SG_CUDA(cudaStreamWaitEvent(gs, m->graph_event, 0));
    g = &m->graphs[m->graph_next];
    m->graph_next = (m->graph_next + 1) % 4;
    free_graph_slot(*g);
    SG_CUDA(cudaMallocHost(&g->hR, sizeof(double) * n_geo * dimi));
    SG_CUDA(cudaMallocHost(&g->hF, sizeof(double) * n_geo * dimi));
    SG_CUDA(cudaMallocHost(&g->hE, sizeof(double) * n_geo));
    std::copy(R, R + n_geo * dimi, g->hR);
    // first call: run the sequence un-captured (sets the kernels' shared-memory attributes) ...
    SG_TRY(enqueue(g));
    SG_CUDA(cudaStreamSynchronize(gs));
    // ... then capture it
    long long before = 0, after = 0;
    for (int k = 0; k < KID_COUNT; ++k) {
      int64_t ln = 0;
      sgdml_b200_profile_get(k, nullptr, nullptr, &ln);
      before += ln;
    }
    cudaGraph_t graph = nullptr;
    SG_CUDA(cudaStreamBeginCapture(gs, cudaStreamCaptureModeThreadLocal));
    int rc = enqueue(g);
    cudaError_t e = cudaStreamEndCapture(gs, &graph);
    if (rc != 0) {
      if (graph) cudaGraphDestroy(graph);
      return rc;
    }
    SG_CUDA(e);
    e = cudaGraphInstantiate(&g->exec, graph, 0);
    cudaGraphDestroy(graph);
    SG_CUDA(e);
    for (int k = 0; k < KID_COUNT; ++k) {
      int64_t ln = 0;
      sgdml_b200_profile_get(k, nullptr, nullptr, &ln);
      after += ln;
    }
    g->n_kernels = (int)(after - before);
    g->n_geo = n_geo;
    g->with_E = with_E;
    g->generation = m->generation;
  } else {
    // replay on the CALLER's stream: ordered after whatever it has queued, no event round trip
    std::copy(R, R + n_geo * dimi, g->hR);
    SG_CUDA(cudaGraphLaunch(g->exec, s));
    count_launch(KID_PREDICT_AUX, g->n_kernels);  // the kernels of a replay are launches too
    SG_CUDA(cudaStreamSynchronize(s));
  }
  std::copy(g->hF, g->hF + n_geo * dimi, F);
  if (with_E) std::copy(g->hE, g->hE + n_geo, E);
  return 0;
}

}  // namespace

int sgdml_b200_model_destroy(sgdml_b200_model* m) {
  if (m == nullptr) return 0;
  cudaDeviceSynchronize();  // the device blocks go back to the cache: no kernel of this model may still run
  for (auto& g : m->graphs) free_graph_slot(g);
  if (m->graph_stream) cudaStreamDestroy(m->graph_stream);
  if (m->graph_event) cudaEventDestroy(m->graph_event);
  cached_free(m->X);
  cached_free(m->Xc);
  cached_free(m->JA);
  cached_free(m->mm);
  cached_free(m->xja);
  cached_free(m->ae);
  cached_free(m->mu);
  cached_free(m->perm);
  cached_free(m->pinv);
  cached_free(m->R_d_desc);
  cached_free(m->XcT);
  cached_free(m->JAT);
  free_oz(m->ozXc);
  free_oz(m->ozJA);
  free_oz(m->ozXcT);
  free_oz(m->ozJAT);
  free_ws(m);
  for (int i = 0; i < 2; ++i)
    if (m->pipe_stream[i]) cudaStreamDestroy(m->pipe_stream[i]);
  for (int i = 0; i < 3; ++i)
    if (m->pipe_event[i]) cudaEventDestroy(m->pipe_event[i]);
  delete m;
  return 0;
}

int sgdml_b200_predict(sgdml_b200_model* m, const double* R, int64_t n_geo, double* E, double* F, void* stream) {
  SG_TRY(require_device());
  SG_ARG(m != nullptr && R != nullptr && F != nullptr && n_geo >= 0);
  if (n_geo == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const bool R_dev = is_device_ptr(R), F_dev = is_device_ptr(F), E_dev = (E != nullptr) && is_device_ptr(E);
  const bool host_io = !R_dev || !F_dev || (E != nullptr && !E_dev);
  const int dimi = 3 * m->N;
  if (!R_dev && !F_dev && (E == nullptr || !E_dev) && n_geo <= GRAPH_MAX_GEO && !profiling_enabled() &&
      g_graph_enabled())
    return predict_graph(m, R, n_geo, E, F, s);
  int64_t chunk = std::min<int64_t>(chunk_geos(m), n_geo);
  // Host buffers: split the batch into >= 4 chunks and run them on two side streams so that the
  // H2D copy of chunk k+1 and the D2H copy of chunk k-1 overlap the kernels of chunk k.
  const bool pipelined = host_io && n_geo >= 4096 && !profiling_enabled();
  if (pipelined) chunk = std::min<int64_t>(chunk, std::max<int64_t>(1024, (n_geo + 3) / 4));
  SG_TRY(ensure_ws(m, 0, chunk));
  if (pipelined) {
    SG_TRY(ensure_ws(m, 1, chunk));
    SG_TRY(ensure_pipe(m));
    SG_CUDA(cudaEventRecord(m->pipe_event[2], s));
    SG_CUDA(cudaStreamWaitEvent(m->pipe_stream[0], m->pipe_event[2], 0));
    SG_CUDA(cudaStreamWaitEvent(m->pipe_stream[1], m->pipe_event[2], 0));
  }
  int c_idx = 0;
  for (int64_t g0 = 0; g0 < n_geo; g0 += chunk, ++c_idx) {
    const int slot = pipelined ? (c_idx & 1) : 0;
    cudaStream_t st = pipelined ? m->pipe_stream[slot] : s;
    sgdml_b200_model::WS& w = m->ws[slot];
    const int64_t ng = std::min<int64_t>(chunk, n_geo - g0);
    const double* Rd = R + g0 * dimi;
    if (!R_dev) {
      SG_CUDA(cudaMemcpyAsync(w.R, Rd, sizeof(double) * ng * dimi, cudaMemcpyHostToDevice, st));
      Rd = w.R;
    }
    SG_TRY(launch_desc_from_R(Rd, ng, m->N, w.xq, w.gq, st, &m->lat));
    double* Fd = F_dev ? F + g0 * dimi : w.F;
    double* Ed = (E == nullptr) ? nullptr : (E_dev ? E + g0 : w.E);
    SG_TRY(run_queries(m, slot, w.xq, w.gq, ng, m->std, m->c, Ed, Fd, st));
    if (!F_dev) SG_CUDA(cudaMemcpyAsync(F + g0 * dimi, Fd, sizeof(double) * ng * dimi, cudaMemcpyDeviceToHost, st));
    if (E != nullptr && !E_dev) SG_CUDA(cudaMemcpyAsync(E + g0, Ed, sizeof(double) * ng, cudaMemcpyDeviceToHost, st));
  }
  if (pipelined) {
    for (int i = 0; i < 2; ++i) {
      SG_CUDA(cudaEventRecord(m->pipe_event[i], m->pipe_stream[i]));
      SG_CUDA(cudaStreamWaitEvent(s, m->pipe_event[i], 0));
    }
  }
  if (host_io) SG_CUDA(cudaStreamSynchronize(s));
  return 0;
}

// Analytic Hessian (csrc/hessian.cu).  Per chunk of queries: descriptors, the predictor's run_queries (E, F and the
// descriptor-space force rows G), then the Hessian kernels on the query rows it leaves in the workspace.
int sgdml_b200_predict_hessian(sgdml_b200_model* m, const double* R, int64_t n_geo, double* E, double* F, double* H,
                               void* stream) {
  SG_TRY(require_device());
  SG_ARG(m != nullptr && R != nullptr && H != nullptr && n_geo >= 0);
  if (n_geo == 0) return 0;
  if ((size_t)m->D * 8 > 200 * 1024) {  // the limit of the predictor's finishing kernel
    set_last_error("sgdml_b200_predict_hessian: molecule too large (n_atoms <= ~225 supported)");
    return SGDML_B200_ERR_UNSUPPORTED;
  }
  cudaStream_t s = (cudaStream_t)stream;
  const bool R_dev = is_device_ptr(R), H_dev = is_device_ptr(H);
  const bool F_dev = F != nullptr && is_device_ptr(F), E_dev = E != nullptr && is_device_ptr(E);
  const int dimi = 3 * m->N;
  const int64_t hsz = (int64_t)dimi * dimi;
  HessModel hm;
  hm.N = m->N;
  hm.D = m->D;
  hm.DS = m->DS;
  hm.M = m->M;
  hm.S = m->S;
  hm.Mpad = m->Mpad;
  hm.sig = m->sig;
  hm.std = m->std;
  hm.X = m->X;
  hm.Xc = m->Xc;
  hm.JA = m->JA;
  hm.mm = m->mm;
  hm.xja = m->xja;
  hm.ae = m->use_ae ? m->ae : nullptr;
  hm.perm = m->perm;
  const int64_t chunk = std::min<int64_t>(n_geo, std::min<int64_t>(chunk_geos(m), hessian_chunk_geos(hm)));
  SG_TRY(ensure_ws(m, 0, chunk));
  sgdml_b200_model::WS& w = m->ws[0];
  // one device block for the Hessian workspace (+ the output staging of host H), back to the cache at the end
  const int64_t last = n_geo - (n_geo - 1) / chunk * chunk;
  const size_t ws_bytes = std::max(hessian_workspace_bytes(hm, chunk), hessian_workspace_bytes(hm, last));
  const size_t stage_bytes = H_dev ? 0 : (size_t)chunk * hsz * 8;
  char* hws = nullptr;
  SG_CUDA(cached_malloc(&hws, ws_bytes + stage_bytes));
  auto body = [&]() -> int {
    for (int64_t g0 = 0; g0 < n_geo; g0 += chunk) {
      const int64_t ng = std::min<int64_t>(chunk, n_geo - g0);
      const double* Rd = R + g0 * dimi;
      if (!R_dev) {
        SG_CUDA(cudaMemcpyAsync(w.R, Rd, sizeof(double) * ng * dimi, cudaMemcpyHostToDevice, s));
        Rd = w.R;
      }
      SG_TRY(launch_desc_from_R(Rd, ng, m->N, w.xq, w.gq, s, &m->lat));
      double* Fd = F_dev ? F + g0 * dimi : w.F;
      double* Ed = (E == nullptr) ? nullptr : (E_dev ? E + g0 : w.E);
      int n_splits = 1;
      SG_TRY(run_queries(m, 0, w.xq, w.gq, ng, m->std, m->c, Ed, Fd, s, &n_splits, true));
      HessChunk hc;
      hc.ng = ng;
      hc.xq = w.xq;
      hc.gq = w.gq;
      hc.Qg = w.Qg;
      hc.qq = w.qq;
      hc.G = w.G;
      hc.DP = m->DP;
      hc.n_splits_G = n_splits;
      hc.plane_rows = (ng * m->S + m->BQ - 1) / m->BQ * m->BQ;
      hc.H = H_dev ? H + g0 * hsz : reinterpret_cast<double*>(hws + ws_bytes);
      SG_TRY(run_hessian(hm, hc, hws, s));
      if (F != nullptr && !F_dev)
        SG_CUDA(cudaMemcpyAsync(F + g0 * dimi, Fd, sizeof(double) * ng * dimi, cudaMemcpyDeviceToHost, s));
      if (E != nullptr && !E_dev) SG_CUDA(cudaMemcpyAsync(E + g0, Ed, sizeof(double) * ng, cudaMemcpyDeviceToHost, s));
      if (!H_dev) SG_CUDA(cudaMemcpyAsync(H + g0 * hsz, hc.H, sizeof(double) * ng * hsz, cudaMemcpyDeviceToHost, s));
    }
    return 0;
  };
  const int rc = body();
  cudaError_t e = cudaStreamSynchronize(s);  // the workspace block goes back to the cache: nothing may still use it
  cached_free(hws);
  if (rc != 0) return rc;
  SG_CUDA(e);
  return 0;
}

int sgdml_b200_model_set_lattice(sgdml_b200_model* m, const double* lattice, const double* lattice_inv) {
  SG_ARG(m != nullptr);
  SG_CUDA(cudaDeviceSynchronize());  // no stream argument: kernels in flight copied the old cell by value, but keep calls ordered
  ++m->generation;  // captured graphs carry the cell as a kernel argument
  return lattice_from_host(lattice, lattice_inv, &m->lat);
}

int sgdml_b200_model_set_alphas_E(sgdml_b200_model* m, const double* alphas_E, void* stream) {
  SG_TRY(require_device());
  SG_ARG(m != nullptr);
  cudaStream_t s = (cudaStream_t)stream;
  ++m->generation;  // captured graphs carry use_ae as a kernel argument
  if (alphas_E == nullptr) {
    SG_CUDA(cudaMemsetAsync(m->ae, 0, sizeof(double) * m->Mpad, s));
    m->use_ae = 0;
    return 0;
  }
  SG_CUDA(cudaMemcpyAsync(m->ae, alphas_E, sizeof(double) * m->M, cudaMemcpyDefault, s));
  if (!is_device_ptr(alphas_E)) SG_CUDA(cudaStreamSynchronize(s));
  m->use_ae = 1;
  return 0;
}

int sgdml_b200_model_set_R_d_desc(sgdml_b200_model* m, const double* R_d_desc) {
  SG_TRY(require_device());
  SG_ARG(m != nullptr && R_d_desc != nullptr);
  const size_t bytes = sizeof(double) * (size_t)m->M * m->D * 3;
  // this entry point has no stream argument: order it against work the caller may have in flight on ANY
  // stream (k_set_alphas / predict kernels of a non-blocking torch stream read m->R_d_desc)
  SG_CUDA(cudaDeviceSynchronize());
  if (m->R_d_desc == nullptr) SG_CUDA(cached_malloc(&m->R_d_desc, bytes));
  SG_CUDA(cudaMemcpy(m->R_d_desc, R_d_desc, bytes, cudaMemcpyDefault));
  SG_CUDA(cudaDeviceSynchronize());
  return 0;
}

int sgdml_b200_model_set_alphas(sgdml_b200_model* m, const double* alphas_F, void* stream) {
  SG_TRY(require_device());
  SG_ARG(m != nullptr && alphas_F != nullptr);
  if (m->R_d_desc == nullptr) {
    set_last_error("sgdml_b200_model_set_alphas: call sgdml_b200_model_set_R_d_desc first (predict.py:575)");
    return SGDML_B200_ERR_ARG;
  }
  cudaStream_t s = (cudaStream_t)stream;
  Staged sA;
  SG_TRY(sA.init(alphas_F, sizeof(double) * (size_t)m->M * 3 * m->N, true, s));
  const int64_t tot = (int64_t)m->M * m->D;
  k_set_alphas<<<ceil_div(tot, 256), 256, 0, s>>>(m->R_d_desc, (const double*)sA.dev(), m->M, m->D, m->N, m->DS,
                                                  m->JA);
  SG_CUDA(cudaGetLastError());
  count_launch(KID_PREDICT_AUX);
  SG_TRY(refresh_row_dots(m, false, s));
  if (m->large) {
    SG_TRY(refresh_transposes(m, false, s));
    SG_TRY(refresh_oz_model(m, false, s));
  }
  if (sA.staged()) SG_CUDA(cudaStreamSynchronize(s));
  return 0;
}

int sgdml_b200_predict_train(sgdml_b200_model* m, int64_t m_begin, int64_t m_end, int scaled, double* E, double* F,
                             void* stream) {
  SG_TRY(require_device());
  SG_ARG(m != nullptr && F != nullptr);
  SG_ARG(m_begin >= 0 && m_end <= m->M && m_begin <= m_end);
  if (m->R_d_desc == nullptr) {
    set_last_error("sgdml_b200_predict_train: call sgdml_b200_model_set_R_d_desc first (predict.py:1223-1229)");
    return SGDML_B200_ERR_ARG;
  }
  const int64_t n_geo = m_end - m_begin;
  if (n_geo == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t chunk = std::min<int64_t>(chunk_geos(m), n_geo);
  SG_TRY(ensure_ws(m, 0, chunk));
  sgdml_b200_model::WS& w = m->ws[0];
  const bool F_dev = is_device_ptr(F), E_dev = (E != nullptr) && is_device_ptr(E);
  const int dimi = 3 * m->N;
  const double std = scaled ? m->std : 1.0, c = scaled ? m->c : 0.0;
  for (int64_t g0 = 0; g0 < n_geo; g0 += chunk) {
    const int64_t ng = std::min<int64_t>(chunk, n_geo - g0);
    const double* xq = m->X + (m_begin + g0) * m->D;
    const double* gq = m->R_d_desc + (m_begin + g0) * m->D * 3;
    double* Fd = F_dev ? F + g0 * dimi : w.F;
    double* Ed = (E == nullptr) ? nullptr : (E_dev ? E + g0 : w.E);
    SG_TRY(run_queries(m, 0, xq, gq, ng, std, c, Ed, Fd, s));
    if (!F_dev) SG_CUDA(cudaMemcpyAsync(F + g0 * dimi, Fd, sizeof(double) * ng * dimi, cudaMemcpyDeviceToHost, s));
    if (E != nullptr && !E_dev) SG_CUDA(cudaMemcpyAsync(E + g0, Ed, sizeof(double) * ng, cudaMemcpyDeviceToHost, s));
  }
  if (!F_dev || (E != nullptr && !E_dev)) SG_CUDA(cudaStreamSynchronize(s));
  return 0;
}

int sgdml_b200_model_set_contraction_slices(sgdml_b200_model* m, int slices, void* stream) {
  SG_ARG(m != nullptr && (slices == 0 || (slices >= 2 && slices <= 7)));
  if (!m->large) return 0;  // D <= 256: the fused FP64 kernel, nothing to choose
  if (slices >= 2 && !(m->DS <= (1 << 14) && m->Mpad <= (1 << 14))) slices = 0;
  if (slices == m->oz_s) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  free_ws(m);  // (synchronises) the per-batch workspaces carry slice buffers sized for the old setting
  ++m->generation;
  m->oz_s = slices;
  if (slices >= 2) {
    SG_TRY(refresh_oz_model(m, true, s));
  } else {
    free_oz(m->ozXc);
    free_oz(m->ozJA);
    free_oz(m->ozXcT);
    free_oz(m->ozJAT);
  }
  return 0;
}

int sgdml_b200_set_predict_variant(int variant) {
  SG_ARG(variant >= 0 && variant <= 5);
  g_predict_variant = variant;
  return 0;
}

int sgdml_b200_model_dims(const sgdml_b200_model* m, int64_t* n_atoms, int64_t* n_train, int64_t* n_perms) {
  SG_ARG(m != nullptr);
  if (n_atoms) *n_atoms = m->N;
  if (n_train) *n_train = m->M;
  if (n_perms) *n_perms = m->S;
  return 0;
}

int sgdml_b200_model_get_R_d_desc_alpha(sgdml_b200_model* m, double* out) {
  SG_TRY(require_device());
  SG_ARG(m != nullptr && out != nullptr);
  SG_CUDA(cudaDeviceSynchronize());  // no stream argument: wait for set_alphas kernels on the caller's streams
  Staged sO;
  SG_TRY(sO.init(out, sizeof(double) * (size_t)m->M * m->D, false, 0));
  const int64_t tot = (int64_t)m->M * m->D;
  k_unpad_rows<<<ceil_div(tot, 256), 256, 0, 0>>>(m->JA, m->M, m->D, m->DS, (double*)sO.dev());
  SG_CUDA(cudaGetLastError());
  SG_TRY(sO.finish(0));
  SG_CUDA(cudaStreamSynchronize(0));
  return 0;
}

}  // extern "C"
