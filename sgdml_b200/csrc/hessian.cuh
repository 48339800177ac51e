// Internal interface of the analytic Hessian kernels (hessian.cu), driven by sgdml_b200_predict_hessian in predict.cu.
#pragma once
#include "common.cuh"

namespace sgdml {

// device views of the predictor's model arrays (struct sgdml_b200_model, predict.cu)
struct HessModel {
  int N, D, DS, M, S, Mpad;
  double sig, std;
  const double* X;    // (M, D) raw training descriptors
  const double* Xc;   // (Mpad, DS) centred, zero padded
  const double* JA;   // (Mpad, DS) R_d_desc_alpha, zero padded
  const double* mm;   // (Mpad) |Xc_m|^2
  const double* xja;  // (Mpad) Xc_m . JA_m
  const double* ae;   // (Mpad) alphas_E, or nullptr
  const int* perm;    // (S, D)
};

// one chunk of ng queries after run_queries (predict.cu) has run on it
struct HessChunk {
  int64_t ng;
  const double* xq;     // (ng, D) query descriptors
  const double* gq;     // (ng, D, 3) compressed query Jacobians
  const double* Qg;     // (ng*S rows, DS) virtual query rows
  const double* qq;     // (ng*S) |Qg row|^2
  const double* G;      // descriptor-space force rows of the predictor, n_splits_G planes of plane_rows x DP
  int DP, n_splits_G;
  int64_t plane_rows;
  double* H;            // (ng, 3N, 3N) device output
};

// queries per chunk: the Hessian workspace of a chunk stays within ~256 MB
int64_t hessian_chunk_geos(const HessModel& hm);
// device workspace (bytes) for a chunk of ng queries
size_t hessian_workspace_bytes(const HessModel& hm, int64_t ng);
// weights, Gram, finish for one chunk; stream-ordered, no allocation (ws: hessian_workspace_bytes(hm, c.ng) bytes)
int run_hessian(const HessModel& hm, const HessChunk& c, void* ws, cudaStream_t s);

}  // namespace sgdml
