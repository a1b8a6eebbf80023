// Internal interface of mvt.cu: the pieces the sqrtm (mvt.cu) and Cholesky (mvt_chol.cu) reparameterisations of the
// full-rank MultivariateT family share.  Both see the same |z_s / u_s|^2 Mahalanobis term at a reparameterised
// sample, so the per-sample weights, the objective value and the mean gradient are the same kernels.
#pragma once
#include "common.cuh"

namespace vb {

// log Gamma((df + d) / 2) - log Gamma(df / 2) - d/2 log(pi df): the df-only part of multivariate_t_logpdf
inline double mvt_const(double df, int d) {
  return lgamma(0.5 * (df + d)) - lgamma(0.5 * df) - 0.5 * d * log(3.14159265358979323846 * df);
}

// one m8n8k4 float64 MMA (DMMA) on the fragment (c0, c1) += a b
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// offset of row i of a packed row-major lower triangle
__host__ __device__ __forceinline__ int64_t tri(int64_t i) { return i * (i + 1) / 2; }

// inv_u[s] = 1 / sqrt(chi2_s / df),  zu2[s] = |z_s / u_s|^2
int mvt_rows(const double* z, const double* chi2, double df, int S, int d, double* inv_u, double* zu2, cudaStream_t stream);

// out[0] = sum_i F_ii (= 0.5 log det Sigma) from var_param
int mvt_logdiag(const double* var_param, int d, double* out, cudaStream_t stream);

// Sample weights sv[S] (1 for ExclusiveKL), scal = {value, diag_add}, value[0] = scal[0] and gmu[d] = c sum_s sv_s G[s]
// with c = -1/S (ExclusiveKL) or alpha/S (AlphaDivergence).
int mvt_weights_gmu(const double* f, const double* G, const double* zu2, const double* half_logdet, int S, int d, double df,
                    int objective, double alpha, double* sv, double* scal, double* value, double* gmu, cudaStream_t stream);

}  // namespace vb
