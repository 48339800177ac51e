// Analytic Hessian H = d^2 E / dR^2 of a GDML model (no counterpart in the reference, which stops at forces).
//
// Per query x (descriptor, length D, Jacobian J = dx/dR) and virtual row (m, p) -- training point m, permutation p,
// delta = x - X_m[perm_p], n = sqrt5 |delta|, base = exp(-n/sig) 5/(3 sig^3), a = delta . JA_m[perm_p]:
//   w_I  = (5/sig) a base         [+ ae base (n + sig)]
//   w_uv = 5 base / sig
//   w_uu = -25 a base / (sig^2 n) [- ae 5 base / sig]        (0 at n = 0: the limit, |a delta delta^T / n| <= |JA| |delta|^2)
//   u = J^T delta,  v = J^T JA_m[perm_p]                      (3N each)
//   H = -std [ (sum w_I) J^T J + sum_(m,p) (w_uv (u v^T + v u^T) + w_uu u u^T) + sum_d Fd_d d^2 x_d / dR^2 ]
// with Fd the descriptor-space force of the predictor (DESIGN.md, "Hessian").
//
// Kernels:
//  * S1 = Q Xc^T, S2 = Q JA^T: the DMMA GEMM of solve.cu (k = DS), always FP64;
//  * k_hess_weights: (S1, S2) -> (w_uu, w_uv) in place, sum_m w_I per virtual row (GEMM-form distance as in
//    k_transform_rows of predict.cu);
//  * k_hess_gram (the hot path): one CTA per (query, 64 x 64 lower tile (I, J) of H, range of training points).
//    For each block of 32 (m, p) pairs the CTA builds u, v on the tile's coordinates -- a sparse J^T product,
//    2 (N - 1) terms per atom -- into shared memory and accumulates A^T B on the FP64 tensor pipe
//    (mma.sync m8n8k4.f64), A = [u; v], B = [w_uu u + w_uv v; w_uv u] over the 64 rows of the block.  Small batches
//    split the pairs into partial planes (summed in fixed order by the finishing kernel: no atomics);
//  * k_hess_fd: the descriptor-space force Fd of each query, a fold of the predictor's G rows through perm;
//  * k_hess_finish: + (sum w_I) J^T J + sum_d Fd_d B_d, times -std, lower tile mirrored -> full (3N, 3N).
#include <algorithm>
#include <cmath>

#include "desc.cuh"
#include "hessian.cuh"
#include "solve.cuh"

namespace sgdml {

namespace {

constexpr int HT = 64;         // H tile edge (coordinates)
constexpr int HLD = HT + 4;    // shared row stride, == 4 mod 16: conflict-free DMMA fragment loads
constexpr int HNP = 32;        // (training point, permutation) pairs per block
constexpr int HK = 2 * HNP;    // contraction rows per block: u and v of every pair
constexpr int HNT = 256;
constexpr int STAGE_D_MAX = 2048;  // query descriptor + Jacobian staged in shared memory up to this D (N <= 64)
constexpr size_t HESS_WS_CAP = 256ull << 20;

inline int n_tiles_side(int N) { return (3 * N + HT - 1) / HT; }
inline int n_tile_pairs(int N) {
  const int T = n_tiles_side(N);
  return T * (T + 1) / 2;
}

__device__ __forceinline__ void tile_pair(int t, int& I, int& J) {  // t = I (I + 1) / 2 + J, J <= I
  int i = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
  while (i * (i + 1) / 2 > t) --i;
  while ((i + 1) * (i + 2) / 2 <= t) ++i;
  I = i;
  J = t - i * (i + 1) / 2;
}

// One warp per virtual row r = (b, p): S1[r][m] -> w_uu, S2[r][m] -> w_uv (zero for padded m), csum[r] = sum_m w_I.
// x5 = 5 |delta|^2 in GEMM form (5 (|q|^2 + |Xc_m|^2 - 2 q.Xc_m)); below 1e-12 of its terms it is cancellation noise
// and the row is taken as n = 0 (w_uu = 0, its limit).
__global__ void __launch_bounds__(256) k_hess_weights(double* __restrict__ S1, double* __restrict__ S2, int64_t ldS,
                                                      const double* __restrict__ qq, const double* __restrict__ mm,
                                                      const double* __restrict__ xja, const double* __restrict__ ae,
                                                      int M, int Mpad, int64_t n_rows, double sig,
                                                      double* __restrict__ csum) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  double* s1 = S1 + r * ldS;
  double* s2 = S2 + r * ldS;
  const double q5 = 5.0 * qq[r];
  const double k_base = 5.0 / (3.0 * sig * sig * sig);
  const double sig_inv = 1.0 / sig;
  double cs = 0.0;
  for (int m = lane; m < Mpad; m += 32) {
    double wuu = 0.0, wuv = 0.0;
    if (m < M) {
      const double t5 = q5 + 5.0 * mm[m];
      const double x5 = fma(-10.0, s1[m], t5);
      const double a = s2[m] - xja[m];
      const bool zero = !(x5 > 1e-12 * t5);
      const double nrm = zero ? 0.0 : sqrt(x5);
      const double base = exp(-nrm * sig_inv) * k_base;
      double wI = a * base * (5.0 * sig_inv);
      wuv = base * (5.0 * sig_inv);
      wuu = zero ? 0.0 : -25.0 * a * base * sig_inv * sig_inv / nrm;
      if (ae != nullptr) {
        wI = fma(ae[m], base * (nrm + sig), wI);
        wuu = fma(-ae[m], wuv, wuu);
      }
      cs += wI;
    }
    s1[m] = wuu;
    s2[m] = wuv;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cs += __shfl_xor_sync(0xffffffffu, cs, o);
  if (lane == 0) csum[r] = cs;
}

struct GramArgs {
  const double* X;    // (M, D)
  const double* JA;   // (Mpad, DS)
  const int* perm;    // (S, D)
  const double* xq;   // (ng, D)
  const double* gq;   // (ng, D, 3)
  const double* Wuu;  // (ng*S, Mpad)
  const double* Wuv;
  int N, D, DS, M, S, Mpad, TP;
  int64_t ng;
  int n_blk, blk_per_split, stage_q;
  double* Hpart;      // [split][b][tile pair][HT*HT]
};

// u, v of atom k (3 components each) for the pair (m, p): sum over the N - 1 partners of +-g_d (x_d - X_m[e]),
// +-g_d JA_m[e], e = perm_p[d]; J[d, a] = -g_d, J[d, b] = +g_d for d = (a, b), a > b
__device__ __forceinline__ void atom_uv(const GramArgs& p, const double* __restrict__ x, const double* __restrict__ g,
                                        int k, int m, int pp, double u[3], double v[3]) {
  const int* __restrict__ pr = p.perm + (int64_t)pp * p.D;
  const double* __restrict__ Xm = p.X + (int64_t)m * p.D;
  const double* __restrict__ Jm = p.JA + (int64_t)m * p.DS;
  u[0] = u[1] = u[2] = v[0] = v[1] = v[2] = 0.0;
  const int dk = k * (k - 1) / 2;
  for (int o = 0; o < k; ++o) {  // k is the larger atom of the pair: -g
    const int d = dk + o;
    const int e = __ldg(pr + d);
    const double dx = __ldg(Xm + e) - x[d];
    const double ja = -__ldg(Jm + e);
    const double g0 = g[3 * d], g1 = g[3 * d + 1], g2 = g[3 * d + 2];
    u[0] = fma(g0, dx, u[0]);
    u[1] = fma(g1, dx, u[1]);
    u[2] = fma(g2, dx, u[2]);
    v[0] = fma(g0, ja, v[0]);
    v[1] = fma(g1, ja, v[1]);
    v[2] = fma(g2, ja, v[2]);
  }
  int d = k * (k + 1) / 2 + k;  // pair (k + 1, k)
  for (int o = k + 1; o < p.N; ++o) {  // k is the smaller atom: +g
    const int e = __ldg(pr + d);
    const double dx = x[d] - __ldg(Xm + e);
    const double ja = __ldg(Jm + e);
    const double g0 = g[3 * d], g1 = g[3 * d + 1], g2 = g[3 * d + 2];
    u[0] = fma(g0, dx, u[0]);
    u[1] = fma(g1, dx, u[1]);
    u[2] = fma(g2, dx, u[2]);
    v[0] = fma(g0, ja, v[0]);
    v[1] = fma(g1, ja, v[1]);
    v[2] = fma(g2, ja, v[2]);
    d += o;  // pair (o + 1, k) = pair (o, k) + o
  }
}

__global__ void __launch_bounds__(HNT) k_hess_gram(const GramArgs p) {
  extern __shared__ __align__(16) double hsm[];
  double* LI = hsm;                 // [HK][HLD]: rows (u, v) of each pair on the tile-I coordinates
  double* RJ = LI + HK * HLD;       // [HK][HLD]: rows (w_uu u + w_uv v, w_uv u) on the tile-J coordinates
  double* wsm = RJ + HK * HLD;      // [2][HNP]: w_uu, w_uv of the block's pairs
  double* qs = wsm + 2 * HNP;       // staged query: x (D), g (3D)

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int lr = lane >> 2, lc = lane & 3;
  const int64_t b = blockIdx.x / p.TP;
  const int t = (int)(blockIdx.x - b * p.TP);
  int I, J;
  tile_pair(t, I, J);
  const bool diag = I == J;
  const int cI = I * HT, cJ = J * HT;
  const int aI0 = cI / 3, natI = min(p.N - 1, (cI + HT - 1) / 3) - aI0 + 1;
  const int aJ0 = cJ / 3, natJ = min(p.N - 1, (cJ + HT - 1) / 3) - aJ0 + 1;

  const double* x = p.xq + b * p.D;
  const double* g = p.gq + b * p.D * 3;
  if (p.stage_q) {
    for (int i = tid; i < p.D; i += HNT) qs[i] = x[i];
    for (int i = tid; i < 3 * p.D; i += HNT) qs[p.D + i] = g[i];
    x = qs;
    g = qs + p.D;
  }
  for (int i = tid; i < 2 * HK * HLD; i += HNT) LI[i] = 0.0;  // coordinates past 3N stay zero
  __syncthreads();

  const int wr = warp >> 1, wc = warp & 1;  // warp tile: rows 16 wr .. +16, columns 32 wc .. +32 of the 64 x 64 tile
  double acc[2][4][2];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

  const int n_pairs = p.M * p.S;
  const int blk0 = (int)blockIdx.y * p.blk_per_split;
  const int blk1 = min(p.n_blk, blk0 + p.blk_per_split);
  const int njobs = HNP * (natI + (diag ? 0 : natJ));
  for (int blk = blk0; blk < blk1; ++blk) {
    const int pair0 = blk * HNP;
    if (tid < HNP) {
      const int pair = pair0 + tid;
      double wuu = 0.0, wuv = 0.0;
      if (pair < n_pairs) {
        const int m = pair / p.S, pp = pair - (pair / p.S) * p.S;
        const int64_t idx = (b * p.S + pp) * p.Mpad + m;
        wuu = p.Wuu[idx];
        wuv = p.Wuv[idx];
      }
      wsm[tid] = wuu;
      wsm[HNP + tid] = wuv;
    }
    __syncthreads();
    // ---- build the block's rows: one job = one (pair, atom) of the tile
    for (int job = tid; job < njobs; job += HNT) {
      const int side = job < HNP * natI ? 0 : 1;
      const int jj = side ? job - HNP * natI : job;
      const int nat = side ? natJ : natI;
      const int jp = jj / nat;
      const int k = (side ? aJ0 : aI0) + (jj - jp * nat);
      const int pair = pair0 + jp;
      double u[3], v[3];
      if (pair < n_pairs) {
        const int m = pair / p.S, pp = pair - m * p.S;
        atom_uv(p, x, g, k, m, pp, u, v);
      } else {
        u[0] = u[1] = u[2] = v[0] = v[1] = v[2] = 0.0;
      }
      const double wuu = wsm[jp], wuv = wsm[HNP + jp];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        if (side == 0) {
          const int col = 3 * k + c - cI;
          if (col >= 0 && col < HT) {
            LI[(2 * jp) * HLD + col] = u[c];
            LI[(2 * jp + 1) * HLD + col] = v[c];
            if (diag) {
              RJ[(2 * jp) * HLD + col] = fma(wuu, u[c], wuv * v[c]);
              RJ[(2 * jp + 1) * HLD + col] = wuv * u[c];
            }
          }
        } else {
          const int col = 3 * k + c - cJ;
          if (col >= 0 && col < HT) {
            RJ[(2 * jp) * HLD + col] = fma(wuu, u[c], wuv * v[c]);
            RJ[(2 * jp + 1) * HLD + col] = wuv * u[c];
          }
        }
      }
    }
    __syncthreads();
    // ---- H_IJ += LI^T RJ on the tensor pipe
    const double* la = LI + lc * HLD + 16 * wr + lr;
    const double* rb = RJ + lc * HLD + 32 * wc + lr;
#pragma unroll 4
    for (int ks = 0; ks < HK / 4; ++ks) {
      double fa[2], fb[4];
#pragma unroll
      for (int i = 0; i < 2; ++i) fa[i] = la[ks * 4 * HLD + 8 * i];
#pragma unroll
      for (int j = 0; j < 4; ++j) fb[j] = rb[ks * 4 * HLD + 8 * j];
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
    }
    __syncthreads();
  }
  double* out = p.Hpart + (((int64_t)blockIdx.y * p.ng + b) * p.TP + t) * (HT * HT);
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
      *reinterpret_cast<double2*>(out + (16 * wr + 8 * i + lr) * HT + 32 * wc + 8 * j + 2 * lc) =
          make_double2(acc[i][j][0], acc[i][j][1]);
}

// Fd[b][d] = sum_p sum_split G_split[b*S + p][perm_p[d]] (the fold of k_predict_finish, unscaled)
__global__ void k_hess_fd(const double* __restrict__ G, const int* __restrict__ perm, int D, int DP, int S,
                          int n_splits, int64_t plane_rows, int64_t ng, double* __restrict__ Fd) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= ng * D) return;
  const int64_t b = idx / D;
  const int d = (int)(idx - b * D);
  const int64_t stride = plane_rows * DP;
  double acc = 0.0;
  for (int pp = 0; pp < S; ++pp) {
    const double* gp = G + (b * S + pp) * DP + perm[pp * D + d];
    for (int sp = 0; sp < n_splits; ++sp) acc += gp[(int64_t)sp * stride];
  }
  Fd[idx] = acc;
}

// One CTA per (query, lower tile): sum of the Gram partial planes (fixed order), + (sum w_I) J^T J + sum_d Fd_d B_d,
// times -std, written to both triangles of the row-major (3N, 3N) output.  With T_d[c][c'] = cs g_c g_c' +
// Fd_d (3 g_c g_c' / x_d - delta_cc' x_d^3)  (x_d = 1/|r|, g_d = r/|r|^3): atom block (k, k) gets sum_o T_d(k,o),
// (k, l != k) gets -T_d(k,l).
__global__ void __launch_bounds__(256) k_hess_finish(const double* __restrict__ Hpart, int n_splits, int TP,
                                                     const double* __restrict__ csum, const double* __restrict__ Fd,
                                                     const double* __restrict__ xq, const double* __restrict__ gq,
                                                     int N, int D, int S, double std, int64_t ng,
                                                     double* __restrict__ H) {
  __shared__ double cs_s;
  const int64_t b = blockIdx.x / TP;
  const int t = (int)(blockIdx.x - b * TP);
  int I, J;
  tile_pair(t, I, J);
  if (threadIdx.x < 32) {
    double s = 0.0;
    for (int pp = threadIdx.x; pp < S; pp += 32) s += csum[b * S + pp];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (threadIdx.x == 0) cs_s = s;
  }
  __syncthreads();
  const double cs = cs_s;
  const int n3 = 3 * N;
  const double* x = xq + b * D;
  const double* g = gq + b * D * 3;
  const double* f = Fd + b * D;
  double* Hb = H + b * n3 * n3;
  const int64_t plane = ng * TP * (HT * HT);
  const double* hp = Hpart + (b * TP + t) * (HT * HT);
  for (int e = threadIdx.x; e < HT * HT; e += blockDim.x) {
    const int i = e / HT, j = e - (e / HT) * HT;
    const int gi = I * HT + i, gj = J * HT + j;
    if (gi >= n3 || gj >= n3 || (I == J && j > i)) continue;
    double s = 0.0;
    for (int sp = 0; sp < n_splits; ++sp) s += hp[sp * plane + e];
    const int k = gi / 3, c = gi - 3 * k;
    const int l = gj / 3, c2 = gj - 3 * l;
    auto T = [&](int d) {
      const double gg = g[3 * d + c] * g[3 * d + c2];
      const double xd = x[d];
      double v = gg * fma(3.0 * f[d], 1.0 / xd, cs);
      if (c == c2) v -= f[d] * xd * xd * xd;
      return v;
    };
    double add = 0.0;
    if (k == l) {
      for (int o = 0; o < N; ++o) {
        if (o == k) continue;
        add += T(o > k ? pair_index(o, k) : pair_index(k, o));
      }
    } else {
      add = -T(k > l ? pair_index(k, l) : pair_index(l, k));
    }
    const double h = -std * (s + add);
    Hb[(int64_t)gi * n3 + gj] = h;
    Hb[(int64_t)gj * n3 + gi] = h;
  }
}

struct Plan {
  int TP, n_blk, splits, blk_per_split;
  size_t off_S2, off_csum, off_Fd, off_Hpart, bytes;
};

size_t align_up(size_t v) { return (v + 255) / 256 * 256; }

Plan make_plan(const HessModel& hm, int64_t ng) {
  Plan pl;
  pl.TP = n_tile_pairs(hm.N);
  pl.n_blk = (int)(((int64_t)hm.M * hm.S + HNP - 1) / HNP);
  const int64_t tile_bytes = (int64_t)HT * HT * 8;
  // small batches: split the (m, p) pairs over CTAs until the grid covers the GPU twice, within the workspace cap
  int64_t sp = (2 * (int64_t)num_sms() + ng * pl.TP - 1) / (ng * pl.TP);
  sp = std::min<int64_t>(sp, (int64_t)HESS_WS_CAP / (ng * pl.TP * tile_bytes));
  sp = std::max<int64_t>(1, std::min<int64_t>(sp, pl.n_blk));
  pl.blk_per_split = (int)((pl.n_blk + sp - 1) / sp);
  pl.splits = (pl.n_blk + pl.blk_per_split - 1) / pl.blk_per_split;
  const size_t rows = (size_t)ng * hm.S;
  const size_t w_bytes = align_up(rows * hm.Mpad * 8);
  pl.off_S2 = w_bytes;
  pl.off_csum = 2 * w_bytes;
  pl.off_Fd = pl.off_csum + align_up(rows * 8);
  pl.off_Hpart = pl.off_Fd + align_up((size_t)ng * hm.D * 8);
  pl.bytes = pl.off_Hpart + (size_t)pl.splits * ng * pl.TP * tile_bytes;
  return pl;
}

}  // namespace

int64_t hessian_chunk_geos(const HessModel& hm) {
  const int64_t n3 = 3 * (int64_t)hm.N;
  // weights, csum, Fd, one Gram plane and the output staging of one query
  const int64_t per_geo = 8 * (2 * (int64_t)hm.S * hm.Mpad + hm.S + hm.D + (int64_t)n_tile_pairs(hm.N) * HT * HT + n3 * n3);
  return std::max<int64_t>(1, std::min<int64_t>(65536, (int64_t)HESS_WS_CAP / per_geo));
}

size_t hessian_workspace_bytes(const HessModel& hm, int64_t ng) { return make_plan(hm, ng).bytes; }

int run_hessian(const HessModel& hm, const HessChunk& c, void* ws, cudaStream_t s) {
  const Plan pl = make_plan(hm, c.ng);
  char* base = static_cast<char*>(ws);
  double* W1 = reinterpret_cast<double*>(base);
  double* W2 = reinterpret_cast<double*>(base + pl.off_S2);
  double* csum = reinterpret_cast<double*>(base + pl.off_csum);
  double* Fd = reinterpret_cast<double*>(base + pl.off_Fd);
  double* Hpart = reinterpret_cast<double*>(base + pl.off_Hpart);
  const int64_t n_rows = c.ng * hm.S;

  // S1 = Q Xc^T, S2 = Q JA^T (FP64 DMMA whatever the model's contraction setting)
  GemmArgs g;
  g.m = n_rows;
  g.n = hm.Mpad;
  g.k = hm.DS;
  g.A = c.Qg;
  g.lda = hm.DS;
  g.ldb = hm.DS;
  g.ldc = hm.Mpad;
  g.alpha = 1.0;
  g.beta = 0.0;
  g.mode = 0;
  g.tri = 0;
  g.abort_flag = nullptr;
  g.B = hm.Xc;
  g.C = W1;
  SG_TRY(launch_gemm(g, s));
  g.B = hm.JA;
  g.C = W2;
  SG_TRY(launch_gemm(g, s));
  {
    ProfScope ps(KID_PREDICT_AUX, s);
    k_hess_weights<<<(unsigned)((n_rows + 7) / 8), 256, 0, s>>>(W1, W2, hm.Mpad, c.qq, hm.mm, hm.xja, hm.ae, hm.M,
                                                                hm.Mpad, n_rows, hm.sig, csum);
    SG_CUDA(cudaGetLastError());
    k_hess_fd<<<(unsigned)((c.ng * hm.D + 255) / 256), 256, 0, s>>>(c.G, hm.perm, hm.D, c.DP, hm.S, c.n_splits_G,
                                                                   c.plane_rows, c.ng, Fd);
    SG_CUDA(cudaGetLastError());
    count_launch(KID_PREDICT_AUX, 2);
  }
  {
    GramArgs a;
    a.X = hm.X;
    a.JA = hm.JA;
    a.perm = hm.perm;
    a.xq = c.xq;
    a.gq = c.gq;
    a.Wuu = W1;
    a.Wuv = W2;
    a.N = hm.N;
    a.D = hm.D;
    a.DS = hm.DS;
    a.M = hm.M;
    a.S = hm.S;
    a.Mpad = hm.Mpad;
    a.TP = pl.TP;
    a.ng = c.ng;
    a.n_blk = pl.n_blk;
    a.blk_per_split = pl.blk_per_split;
    a.stage_q = hm.D <= STAGE_D_MAX ? 1 : 0;
    a.Hpart = Hpart;
    const size_t smem = (size_t)(2 * HK * HLD + 2 * HNP + (a.stage_q ? 4 * hm.D : 0)) * 8;
    static bool configured[64] = {false};
    int dev = 0;
    SG_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !configured[dev]) {
      SG_CUDA(cudaFuncSetAttribute(k_hess_gram, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)((2 * HK * HLD + 2 * HNP + 4 * STAGE_D_MAX) * 8)));
      configured[dev] = true;
    }
    ProfScope ps(KID_HESSIAN, s);
    k_hess_gram<<<dim3((unsigned)(c.ng * pl.TP), (unsigned)pl.splits), HNT, smem, s>>>(a);
    SG_CUDA(cudaGetLastError());
    count_launch(KID_HESSIAN);
  }
  {
    ProfScope ps(KID_PREDICT_AUX, s);
    k_hess_finish<<<(unsigned)(c.ng * pl.TP), 256, 0, s>>>(Hpart, pl.splits, pl.TP, csum, Fd, c.xq, c.gq, hm.N, hm.D,
                                                           hm.S, hm.std, c.ng, c.H);
    SG_CUDA(cudaGetLastError());
    count_launch(KID_PREDICT_AUX);
  }
  return 0;
}

}  // namespace sgdml
