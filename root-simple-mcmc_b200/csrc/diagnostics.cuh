// diagnostics.cuh -- on-device ensemble diagnostics of the accepted points
// (SURVEY.md 8f rank 3).  The reference computes these offline from the output
// TTree, one chain at a time:
//   MakeCovariance.C:63-89        mean_i = sum x_i / N,  cov_ij = sum x_i x_j / N - mean_i mean_j
//   MakeAutocorrelation.C:96-148  a_i(lag) = (<x_i(t) x_i(t-lag)> - mean_i^2) / var_i   ("Pearson" form,
//                                 mean and spread from the TProfile "s" option), on a subset of lags
// Here the sums are accumulated for every chain of the ensemble after every step,
// without the points leaving the GPU, and Gelman-Rubin's R-hat across the chains
// (which a single-chain macro cannot give) comes from the per-chain sums.
//
//   pooled : double[1 + n + n(n+1)/2]   (count, sum x, packed sum x x^T) over chains and steps (kPoolAccumulate)
//   s1, s2 : double[E][n]               per-chain sum x, sum x^2
//   chainCount: double[E]               per-chain number of steps behind s1, s2 (steps it was running)
//   ring   : double[depth][E][n]        the last `depth` accepted points of every chain
//   lagProd: double[nlags][n]           sum over chains and steps of x_i(t) x_i(t - lag)
//   lagCount: double[nlags]             number of (chain, step) pairs behind each lagProd row
#pragma once
#include <cuda_runtime.h>

#include "proposal.cuh"

namespace smcmc {

struct DiagArrays {
    double* pooled;
    double* s1;
    double* s2;
    double* chainCount;
    double* ring;
    double* lagProd;
    double* lagCount;
    const int* lags;
    int nlags;
    int depth;
};

// Per (chain, dimension): per-chain sums and the ring buffer slot of this step.
__global__ void __launch_bounds__(256)
kDiagChains(const double* __restrict__ x, const ChainScalars* __restrict__ sc, int chains, int n,
            DiagArrays d, int slot) {
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= (size_t)chains * n) return;
    const int c = (int)(k / n);
    const bool live = sc == nullptr || (sc[c].started && sc[c].status == 0);
    const double v = live ? x[k] : nan("");
    if (live) {
        d.s1[k] += v;
        d.s2[k] += v * v;
        if (k == (size_t)c * n) d.chainCount[c] += 1.0;
    }
    if (d.depth > 0) d.ring[(size_t)slot * chains * n + k] = v;     // NaN marks a chain that is not running
}

// lagProd[l][i] += sum_c x[c][i] * ring[slot - lag_l][c][i] for every lag already covered by
// the ring buffer.  grid = (blocks over chains x n, nlags); `fills` counts this step.
__global__ void __launch_bounds__(256)
kDiagLags(const double* __restrict__ x, int chains, int n, DiagArrays d, int slot, long long fills) {
    extern __shared__ double dimSum[];       // n sums + 1 count
    const int l = blockIdx.y;
    const int lag = d.lags[l];
    if (fills <= lag) return;
    for (int i = threadIdx.x; i <= n; i += blockDim.x) dimSum[i] = 0.0;
    __syncthreads();
    const size_t total = (size_t)chains * n;
    const int back = (slot - lag % d.depth + d.depth) % d.depth;
    const double* old = d.ring + (size_t)back * total;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (size_t)gridDim.x * blockDim.x) {
        const double a = x[k], b = old[k];
        const int i = (int)(k % n);
        if (!isnan(b) && !isnan(a)) {
            atomicAdd(&dimSum[i], a * b);
            if (i == 0) atomicAdd(&dimSum[n], 1.0);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x)
        if (dimSum[i] != 0.0) atomicAdd(&d.lagProd[(size_t)l * n + i], dimSum[i]);
    if (threadIdx.x == 0 && dimSum[n] != 0.0) atomicAdd(&d.lagCount[l], dimSum[n]);
}

}  // namespace smcmc
