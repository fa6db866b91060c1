// accept_local.cuh -- kAcceptLocal: likelihood of the proposed point AND the tail
// of TSimpleMCMC::Step (:410-495) in one launch, for the likelihoods that need
// only the chain's own point (simple_likelihoods.cuh) and steps without a trace.
//
// kSimpleLikelihood + kAccept read every proposed row twice, one thread per row
// (32 different sectors per load instruction), and write the likelihood to global
// memory in between.  Here a warp owns 32 consecutive chains: their proposed rows
// are ONE contiguous block of 32 n doubles, brought into shared memory by a single TMA
// bulk copy per warp (cp.async.bulk + mbarrier: 12.8 KB in flight per warp at n = 50, no
// address arithmetic; round 1 copied it with four 8-byte loads in flight per lane and an
// integer division per element, and the launch was bound by load latency at a fifth of the
// HBM rate); lane = chain then adds its row in the reference's order from shared memory
// (rows contiguous: an even n costs a 2x bank conflict on the row walk, nothing next to
// the copy), takes the Metropolis decision exactly as kAccept does, and the rows of the
// chains that accepted go to xAcc from the same tile, coalesced.  Same arithmetic, same
// draws: the chains are bit-identical (tests/test_gpu_accept_local.py).
#pragma once
#include "proposal.cuh"
#include "simple_likelihoods.cuh"
#include "smcmc_tma.cuh"

namespace smcmc {

constexpr int kAcceptLocalWarps = 4;
__host__ __device__ inline size_t acceptLocalSmem(int n) {
    return (size_t)kAcceptLocalWarps * 32 * n * sizeof(double);
}

__global__ void __launch_bounds__(kAcceptLocalWarps * 32)
kAcceptLocal(ChainArrays a, PropSettings ps, int chains, int llhKind, uint64_t seed, uint32_t chainOffset,
             StepRef stepRef, int metropolis, const int* __restrict__ acceptSlot /* per chain, or null: slot n */) {
    extern __shared__ __align__(128) double tileAll[];
    __shared__ uint64_t bars[kAcceptLocalWarps];
    const uint32_t step = stepRef.get();
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int n = ps.n;
    double* tile = tileAll + (size_t)warp * 32 * n;
    const int c0 = (blockIdx.x * kAcceptLocalWarps + warp) * 32;
    if (c0 >= chains) return;
    const int nc = min(32, chains - c0);
    const double* src = a.xProp + (size_t)c0 * n;
    const uint32_t bytes = (uint32_t)(nc * n) * (uint32_t)sizeof(double);
    // one bulk copy when source, size and destination are 16-byte multiples (always, for an even
    // number of doubles: c0 is a multiple of 32), else the plain copy
    const bool bulk = ((bytes | (uint32_t)(uintptr_t)src) & 15u) == 0u;
    if (bulk) {
        if (lane == 0) {
            mbarInit(&bars[warp], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            mbarExpectTx(&bars[warp], bytes);
            tmaLoad1D(tile, src, bytes, &bars[warp]);
        }
        __syncwarp();
        mbarWait(&bars[warp], 0);
    } else {
#pragma unroll 4
        for (int k = lane; k < nc * n; k += 32) tile[k] = src[k];
        __syncwarp();
    }
    const int c = c0 + lane;
    bool take = false;
    if (lane < nc) {
        ChainScalars* sp = a.sc + c;
        if (sp->started && sp->status == 0) {
            sp->llhCalls += 1;                                              // :539
            const double* x = tile + lane * n;
            double propLlh;                                                 // :410
            switch (llhKind) {
            case SMCMC_LLH_UNIT_GAUSS: propLlh = llhUnitGauss(x, n); break;
            case SMCMC_LLH_HORRIFIC: propLlh = llhHorrific(x, n); break;
            case SMCMC_LLH_HARD: propLlh = llhHard(x, n); break;
            default: propLlh = llhAsym(x, n); break;
            }
            const double accLlh = sp->accLlh;
            sp->propLlh = propLlh;
            if (metropolis == 2) {                                          // :414-426
                take = true;
            } else if (!devIsFinite(propLlh) || propLlh < -0.999999E+30) {  // :432-436
                take = false;
            } else {
                take = true;
                const double delta = __dsub_rn(propLlh, accLlh);            // :441
                if (delta < 0.0) {
                    if (metropolis == 1) take = false;                      // :448
                    else {
                        const uint32_t slot = acceptSlot ? (uint32_t)acceptSlot[4 * c + 2] : (uint32_t)n;
                        const double uu = __dmul_rn(1.0, smcmc_uniform(seed, chainOffset + (uint32_t)c, step,
                                                                       slot, SMCMC_STREAM_STEP));
                        const double trial = log(uu);                       // :455
                        if (delta < trial) take = false;
                    }
                }
            }
            if (take) sp->accLlh = propLlh;                                 // :484
        }
    }
    // ---- commit: fAccepted = fProposed for the chains that accepted (:485-491) -------
    const unsigned taken = __ballot_sync(0xffffffffu, take);
    if (taken == 0u) return;
    double* dst = a.xAcc + (size_t)c0 * n;
    for (unsigned rows = taken; rows; rows &= rows - 1) {
        const int r = __ffs(rows) - 1;
        for (int i = lane; i < n; i += 32) dst[r * n + i] = tile[r * n + i];
    }
}

}  // namespace smcmc
