// engine.cu -- libsmcmc_b200.so: the engine object behind the C ABI of
// include/smcmc_b200.h.  Host code here only owns device memory, resolves the
// few n-dependent defaults the reference computes once, and queues kernels;
// all per-chain and per-event arithmetic is in the .cuh kernels.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"
#include "contraction.cuh"
#include "diagnostics.cuh"
#include "fake_likelihood.cuh"
#include "hmc.cuh"
#include "hmc_order.h"
#include "nccl_dyn.h"
#include "pooled.cuh"
#include "proposal.cuh"
#include "proposal_staged.cuh"
#include "proposal_resident.cuh"
#include "accept_local.cuh"
#include "simple_likelihoods.cuh"
#include "unbinned_likelihood.cuh"
#include "vaat.cuh"

namespace smcmc {

static thread_local std::string gCreateError;

// Smallest double l with pred(exp(l)) true, for a predicate monotone in l:
// bisection on the ordered bit patterns of positive doubles.
template <class Pred>
static double firstLogWhere(Pred pred, double lo, double hi) {
    // invariant: !pred(exp(lo)), pred(exp(hi)), 0 < lo < hi
    uint64_t a, b;
    std::memcpy(&a, &lo, 8);
    std::memcpy(&b, &hi, 8);
    while (b - a > 1) {
        uint64_t mid = a + (b - a) / 2;
        double m;
        std::memcpy(&m, &mid, 8);
        if (pred(std::exp(m))) b = mid;
        else a = mid;
    }
    double r;
    std::memcpy(&r, &b, 8);
    return r;
}

}  // namespace smcmc

using namespace smcmc;

// Device state of the TSimpleHMC ensemble (hmc.cuh), allocated on first use.
struct HmcHost {
    bool allocated = false, started = false, firstStart = true;
    double alpha = 0.0;              // fAlpha                 TSimpleHMC.H:133
    int userGradient = 0;            // TSimpleHMC<L, L> instead of TSimpleHMC<L>
    int keepError = 0;               // keep fEstimatedError per chain
    DeviceBuffer<double> qAcc, pAcc, qProp, pProp, p0, grad, central, average, exxt, exxtT, estErr, repairedDiag;
    DeviceBuffer<double> llh, fdWork, fdLlh, avgPts, avgLlh;
    DeviceBuffer<double> qAlt, uturn;    // fused leap-frog stage (kHmcLeapDmma): the second q buffer, the U-turn partials
    DeviceBuffer<int> order;             // ... and the chains ordered by trajectory length (ragged ensembles)
    DeviceBuffer<double> gradCur, gradEnd;   // ... the gradients at the accepted and the proposed points (kHmcLeapCached)
    bool gradCacheReady = false;         // gradCur holds the gradient at every running chain's accepted point ...
    int gradCacheMode = -1;              // ... as the path that kept it computes it (gradient kind; 100: fused tensor stage)
    int* hostSteps = nullptr;            // pinned, 2 x chains: the trajectory lengths read back, the order sent
    DeviceBuffer<HmcScalars> sc;
    DeviceBuffer<int> leapSteps, counters, updateList;
    // deferred fEXXT update (hmc.cuh, kHmcExxtFlush): 0 = every step
    DeviceBuffer<double> ring, ringT, exxtDiag;
    DeviceBuffer<int> pending;
    int deferK = 0, sinceFlush = 0;
    // ensemble-pooled covariance (hmc.cuh, kHmcPooled*): -1 automatic, 0 per chain, 1 pooled
    int pooledSetting = -1;
    bool pooled = false;
    DeviceBuffer<int> poolMask;
    DeviceBuffer<double> poolStats, poolExxt, poolAverage, poolDiag, poolScratch, poolLlh;
    DeviceBuffer<HmcPooled> pool;
    int* hostCounters = nullptr;     // pinned
    ~HmcHost() {
        if (hostCounters) cudaFreeHost(hostCounters);
        if (hostSteps) cudaFreeHost(hostSteps);
    }
};

struct smcmc_engine {
    smcmc_config cfg;
    cudaStream_t stream = nullptr;
    std::string lastError;
    int64_t launches = 0;
    int smCount = 148;
    uint32_t stepIndex = 0;
    bool started = false;
    // debugging modes of the proposal (TSimpleMCMC.H:671-704)
    DeviceBuffer<double> forcedStep;    // ForceStep: the next proposal of every chain
    bool forcedPending = false;
    int scanDim = -1;                   // SetScanDimension
    bool vaatInitialized = false;       // TProposeVAATStep::InitializeState ran (it runs once, :197-198)
    // the step loop as a CUDA graph (stepMany): the step counter moves to a device word
    bool graphMode = false;
    DeviceBuffer<uint32_t> dStep;
    cudaStream_t graphStream = nullptr;
    cudaEvent_t graphEvent = nullptr;
    cudaGraphExec_t graphExec = nullptr;
    StepRef stepRef() {
        StepRef r;
        r.value = stepIndex;
        r.ptr = graphMode ? dStep.get() : nullptr;
        return r;
    }

    // ---- proposal settings (host mirror of the reference's members) -------
    std::vector<int> type;
    std::vector<double> param1, param2;
    std::vector<int> corrDim1, corrDim2;
    std::vector<double> corrValue;
    double covWindow = -1, accWindow = -1, target = -1;
    double covDeweight = 0.5, accDeweight = 0.5;
    double maxCorr = 1.0 - std::sqrt(std::numeric_limits<double>::epsilon());
    int covFrozen = 0, stepRMSWindow = 1000;
    bool settingsDirty = true;
    DeviceBuffer<int> dType, dCorr1, dCorr2;
    DeviceBuffer<double> dParam1, dParam2, dCorrValue;

    // ---- per-chain state ---------------------------------------------------
    DeviceBuffer<double> xAcc, xProp, lastPoint, center, cov, decomp, upk, llhProp;
    DeviceBuffer<uint32_t> ijTab;
    int covStride = 0, upkStride = 0;   // doubles per chain (whole 128-byte lines)
    DeviceBuffer<double> fakeTerms;     // kFakeFinish with few points: the 150 bin terms per point
    DeviceBuffer<unsigned int> fakeTickets;
    bool staged = false;                // kProposeStaged (one CTA per chain) instead of kPropose
    bool resident = false;              // kStepsResident fits (whole steps out of shared memory)
    int residentPerSm = 0;              // its CTAs per SM
    int64_t residentLaunches = 0;

    // ---- TProposeVAATStep (vaat.cuh) ---------------------------------------
    int propKind = SMCMC_PROPOSAL_ADAPTIVE;
    bool vaatSynced = false;            // xProp equals xAcc except in the last moved coordinate (vaat.cuh)
    std::vector<double> gaussSigma;     // SetGaussian's argument as given (TProposeVAATStep keeps sigma, not sigma^2)
    int vaatWindow = -1;                // fAcceptanceWindow (int; InitializeState forces 100, TProposeVAATStep.H:208)
    DeviceBuffer<double> vSigma, vAcceptance;
    DeviceBuffer<int> vAccTrials, vQueue;
    DeviceBuffer<VaatState> vState;
    VaatArrays vaatArrays() {
        VaatArrays v;
        v.sigma = vSigma.get();
        v.acceptance = vAcceptance.get();
        v.acceptanceTrials = vAccTrials.get();
        v.queue = vQueue.get();
        v.st = vState.get();
        v.window = vaatWindow;
        v.target = 0.44;                // :30
        return v;
    }
    void vaatAllocate() {
        const size_t En = (size_t)E() * n();
        vSigma.reserve(En);
        vAcceptance.reserve(En);
        vAccTrials.reserve(En);
        vQueue.reserve(En);
        vState.reserve(E());
        std::vector<double> sig(En, 2.34);                                  // SetDim, :95
        CUDA_CHECK(cudaMemcpy(vSigma.get(), sig.data(), En * sizeof(double), cudaMemcpyHostToDevice));
        CUDA_CHECK(cudaMemset(vAcceptance.get(), 0, En * sizeof(double)));
        CUDA_CHECK(cudaMemset(vAccTrials.get(), 0, En * sizeof(int)));
        CUDA_CHECK(cudaMemset(vQueue.get(), 0, En * sizeof(int)));
        std::vector<VaatState> st(E());
        for (auto& q : st) { q.lastIndex = -1; q.queueSize = 0; q.acceptSlot = 0; q.pad_ = 0; }
        CUDA_CHECK(cudaMemcpy(vState.get(), st.data(), st.size() * sizeof(VaatState), cudaMemcpyHostToDevice));
    }
    DeviceBuffer<ChainScalars> sc;
    DeviceBuffer<int32_t> okDev;
    DeviceBuffer<double> eigScratch;
    DeviceBuffer<int> eigLocks;
    int eigSlots = 0;

    // ---- likelihood data ---------------------------------------------------
    smcmc_user_ops userOps = {0, 0, nullptr, nullptr, nullptr};   // USER: the functor's launch table
    DeviceBuffer<double> errMatrix, errMatrixT;     // DUMMY: Error(i,j) row-major, and its transpose
    int errDim = 0;
    int dummyMode = SMCMC_DUMMY_EXACT;              // SMCMC_DUMMY_EXACT | SMCMC_DUMMY_TENSOR
    DeviceBuffer<double> dummyPartials;
    DeviceBuffer<PreparedEvent> fakeEvents;         // FAKE
    DeviceBuffer<FilterTile> fakeFilterTiles;
    DeviceBuffer<FilterChain> fakeFilterChains;
    DeviceBuffer<unsigned long long> fakeStats;
    bool exactOnly = false;
    bool noTileSkip = false;                        // SMCMC_FAKE_NO_SKIP: the pair kernel evaluates every tile
    DeviceBuffer<smcmc_event> fakeIrregular;
    int64_t fakeClassBase[kFakeClasses] = {0, 0, 0, 0};    // padded event index, multiple of kPairTile
    int64_t fakeClassCount[kFakeClasses] = {0, 0, 0, 0};   // events of the class, padding included
    int64_t fakeClassReal[kFakeClasses] = {0, 0, 0, 0};
    int64_t fakeBandStart[kFakeClasses][kMassBands] = {};  // first event of each mass band in its class
    int64_t fakeIrregularCount = 0;
    int64_t fakeEventCount = -1;
    DeviceBuffer<double> fakeData;
    bool fakeDataSet = false;
    double fakeExposure = 1.0;
    DeviceBuffer<FakeChainParams> fakeChains;
    DeviceBuffer<uint32_t> fakeCounts;
    int fakeCountStride = 0;
    bool forceGeneric = false;

    // ---- unbinned mixture likelihood (unbinned_likelihood.cuh) ---------------------
    DeviceBuffer<PreparedEvent> unbEvents;
    DeviceBuffer<UnbinnedChain> unbChains;
    DeviceBuffer<double> unbPartial;
    int64_t unbClassCount[2] = {0, 0};
    int64_t unbEventCount = -1;

    // ---- ensemble diagnostics (diagnostics.cuh) ------------------------------------
    bool diagOn = false;
    int diagDepth = 0;
    long long diagFills = 0;
    std::vector<int> diagLags;
    DeviceBuffer<double> diagPooled, diagS1, diagS2, diagChainCount, diagRing, diagLagProd, diagLagCount;
    DeviceBuffer<int> diagLagsDev;

    DiagArrays diagArrays() {
        DiagArrays d;
        d.pooled = diagPooled.get();
        d.s1 = diagS1.get();
        d.s2 = diagS2.get();
        d.chainCount = diagChainCount.get();
        d.ring = diagRing.get();
        d.lagProd = diagLagProd.get();
        d.lagCount = diagLagCount.get();
        d.lags = diagLagsDev.get();
        d.nlags = (int)diagLags.size();
        d.depth = diagDepth;
        return d;
    }
    void diagReset() {
        const size_t En = (size_t)E() * n();
        CUDA_CHECK(cudaMemsetAsync(diagPooled.get(), 0, poolStatCount() * sizeof(double), stream));
        CUDA_CHECK(cudaMemsetAsync(diagS1.get(), 0, En * sizeof(double), stream));
        CUDA_CHECK(cudaMemsetAsync(diagS2.get(), 0, En * sizeof(double), stream));
        CUDA_CHECK(cudaMemsetAsync(diagChainCount.get(), 0, E() * sizeof(double), stream));
        if (!diagLags.empty()) {
            CUDA_CHECK(cudaMemsetAsync(diagLagProd.get(), 0, diagLags.size() * n() * sizeof(double), stream));
            CUDA_CHECK(cudaMemsetAsync(diagLagCount.get(), 0, diagLags.size() * sizeof(double), stream));
        }
        diagFills = 0;
    }
    // the accepted points of this step join the sums (after kAccept)
    void diagAccumulate() {
        const size_t En = (size_t)E() * n();
        DiagArrays d = diagArrays();
        const int slot = diagDepth > 0 ? (int)(diagFills % diagDepth) : 0;
        ++diagFills;
        if (d.nlags > 0) {
            const int blocksX = (int)std::min<size_t>((En + 255) / 256, (size_t)smCount * 4);
            dim3 grid(blocksX, d.nlags);
            kDiagLags<<<grid, 256, (n() + 1) * sizeof(double), stream>>>(xAcc.get(), E(), n(), d, slot, diagFills);
            launched();
        }
        kDiagChains<<<ceilDiv((long long)En, 256), 256, 0, stream>>>(xAcc.get(), sc.get(), E(), n(), d, slot);
        launched();
        poolAccumulate(diagPooled.get());
    }

    // ---- pooled adaptation (pooled.cuh) -----------------------------------------
    int pooledEvery = 0;                            // 0 = per-chain adaptation (the reference)
    DeviceBuffer<double> poolStats, poolStatsAll, poolCov, poolDecomp, poolMean, poolTrace;
    DeviceBuffer<double> poolDecompT, poolZ, poolY;  // TENSOR path of the pooled proposal (n >= 128)
    int pooledTensor = -1;                          // -1: automatic (dim >= 128), 0: off, 1: on
    bool usePooledTensor() const { return pooledTensor < 0 ? n() >= 128 : pooledTensor != 0; }
    void poolTranspose() {
        if (!usePooledTensor()) return;
        const size_t nn = (size_t)n() * n();
        poolDecompT.reserve(nn);
        kTransposeSquare<<<ceilDiv((long long)nn, 256), 256, 0, stream>>>(poolDecomp.get(), poolDecompT.get(), n());
        launched();
    }
    DeviceBuffer<int> poolOk;
    int64_t poolExchanges = 0;

    // ---- multi-GPU (NCCL over NVLink) ---------------------------------------------
    ncclComm_t worldComm = nullptr;                 // pooled-statistics all-reduce
    ncclComm_t eventComm = nullptr;                 // ranks that share chains and split the events
    int worldSize = 1, worldRank = 0, eventGroup = 1;

    PooledState pooled() {
        PooledState p;
        p.stats = poolStats.get();
        p.statsAll = poolStatsAll.get();
        p.cov = poolCov.get();
        p.decomp = poolDecomp.get();
        p.mean = poolMean.get();
        p.trace = poolTrace.get();
        return p;
    }
    int poolStatCount() const { return 1 + n() + tri(); }
    static int poolGramMin() {
        const char* v = std::getenv("SMCMC_POOL_GRAM_MIN");
        return v ? std::atoi(v) : 64;
    }
    // S += the accepted points of the local chains (count, sum x, sum x x^T): Y^T Y on the
    // FP64 tensor cores; SMCMC_POOL_ACC_SCALAR=1 keeps the scalar kernel
    void poolAccumulate(double* stats) { poolAccumulateOn(xAcc.get(), sc.get(), nullptr, stats); }
    // ... of the rows of `x` whose chain is running (scalars) or marked (mask)
    void poolAccumulateOn(const double* x, const ChainScalars* scalars, const int* mask, double* stats) {
        if (!mask && std::getenv("SMCMC_POOL_ACC_SCALAR")) {
            const int poolBlocks = std::min(smCount * 8, ceilDiv(E(), kPoolTile));
            kPoolAccumulate<<<poolBlocks, 256, poolAccSmem(n()), stream>>>(xAcc.get(), sc.get(), E(), n(), stats);
        } else if (n() >= poolGramMin() && !std::getenv("SMCMC_POOL_ACC_DIRECT")) {
            // large dimension: shared-memory tiled Y^T Y (kPoolGramDmma)
            const int nb = ceilDiv(n() + 1, kGramB), pairs = nb * (nb + 1) / 2;
            // chain slices so that the grid is ONE wave of 3 CTAs per SM (13 slices x 36 tile pairs = 468 CTAs
            // on 444 slots ran as two waves: 0.26 ms instead of 0.14 at n = 500)
            int slices = std::max(1, std::min(ceilDiv(E(), 4 * kGramK), (3 * smCount) / pairs));
            slices = std::max(slices, ceilDiv(E(), 4096));                 // the liveness flags of a slice sit in shared memory
            const int perCta = ceilDiv(ceilDiv(E(), slices), kGramK) * kGramK;
            slices = ceilDiv(E(), perCta);
            const size_t smem = kGramSmemBytes + (size_t)((perCta + 15) & ~15);
            if (smem > gramSmemSet) {
                CUDA_CHECK(cudaFuncSetAttribute(kPoolGramDmma<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                CUDA_CHECK(cudaFuncSetAttribute(kPoolGramDmma<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                gramSmemSet = smem;
            }
            if ((n() & 1) == 0)
                kPoolGramDmma<true><<<dim3(pairs, slices), 128, smem, stream>>>(x, scalars, mask, E(), n(), stats, perCta);
            else
                kPoolGramDmma<false><<<dim3(pairs, slices), 128, smem, stream>>>(x, scalars, mask, E(), n(), stats, perCta);
        } else {
            const int blocks = ceilDiv(n() + 1, kPaBlock);
            const int pairs = blocks * (blocks + 1) / 2;
            // three CTAs per SM (168 registers): the loop is bound by load and DMMA latency
            int slices = std::max(1, std::min(ceilDiv(E(), 16), ceilDiv(3 * smCount, pairs)));
            const int perCta = ceilDiv(ceilDiv(E(), slices), 16) * 16;
            slices = ceilDiv(E(), perCta);
            kPoolAccumulateDmma<true><<<dim3(blocks, slices), 128, 0, stream>>>(x, scalars, E(), n(), stats, perCta, mask);
            if (blocks > 1) {
                launched();
                kPoolAccumulateDmma<false><<<dim3(pairs - blocks, slices), 128, 0, stream>>>(x, scalars, E(), n(), stats,
                                                                                         perCta, mask);
            }
        }
        launched();
    }
    static size_t poolAccSmem(int n) { return (size_t)kPoolTile * (n + 2) * sizeof(double); }
    // the tile kernel keeps the shared U and 32 chains in shared memory: four CTAs per SM
    bool usePooledTile() const { return !std::getenv("SMCMC_POOLED_WARP") && pooledTileSmem(n()) <= 56 * 1024; }
    void poolInit() {
        const size_t nn = (size_t)n() * n();
        if (poolAccSmem(n()) > 48 * 1024)
            CUDA_CHECK(cudaFuncSetAttribute(kPoolAccumulate, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)poolAccSmem(n())));
        if (usePooledTile() && pooledTileSmem(n()) > 48 * 1024)
            CUDA_CHECK(cudaFuncSetAttribute(kProposePooledTile, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)pooledTileSmem(n())));
        poolStats.reserve(poolStatCount());
        poolStatsAll.reserve(poolStatCount());
        poolCov.reserve(tri());
        poolDecomp.reserve(2 * nn);
        poolMean.reserve(n());
        poolTrace.reserve(1);
        poolOk.reserve(1);
        CUDA_CHECK(cudaMemsetAsync(poolStats.get(), 0, poolStatCount() * sizeof(double), stream));
        // every chain starts from the same U and trace (same settings): adopt chain 0's
        CUDA_CHECK(cudaMemcpyAsync(poolDecomp.get(), decomp.get(), nn * sizeof(double), cudaMemcpyDeviceToDevice, stream));
        CUDA_CHECK(cudaMemcpyAsync(poolTrace.get(), &sc.get()->sigmaTrace, sizeof(double), cudaMemcpyDeviceToDevice, stream));
        poolTranspose();
    }
    void poolExchange() {
        CUDA_CHECK(cudaMemcpyAsync(poolStatsAll.get(), poolStats.get(), poolStatCount() * sizeof(double),
                                   cudaMemcpyDeviceToDevice, stream));
        if (worldComm) {
            NcclApi& nccl = NcclApi::get();
            nccl.check(nccl.AllReduce(poolStatsAll.get(), poolStatsAll.get(), poolStatCount(), ncclDouble, ncclSum,
                                      worldComm, stream), "all-reduce of pooled statistics");
        }
        if (std::getenv("SMCMC_POOL_FACTOR_WARP")) kPoolFactor<<<1, 32, 0, stream>>>(pooled(), n(), poolOk.get());
        else kPoolFactorCta<<<1, kPoolFactorThreads, 0, stream>>>(pooled(), n(), poolOk.get());
        launched();
        poolTranspose();
        ++poolExchanges;
    }

    // ---- TSimpleHMC ---------------------------------------------------------------
    HmcHost hmc;

    // ---- scratch for smcmc_eval / smcmc_fake_histograms ---------------------
    DeviceBuffer<double> evalX, evalOut, evalHist;

    // ---- instrumentation ----------------------------------------------------
    bool timing = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pairEvents;
    double pairMs = 0.0;
    int64_t pairLaunches = 0;

    int n() const { return cfg.dim; }
    int E() const { return cfg.chains; }
    int tri() const { return cfg.dim * (cfg.dim + 1) / 2; }

    void launched() {
        ++launches;
        CUDA_CHECK(cudaGetLastError());
    }

    ChainArrays arrays() {
        ChainArrays a;
        a.xAcc = xAcc.get();
        a.xProp = xProp.get();
        a.lastPoint = lastPoint.get();
        a.center = center.get();
        a.cov = cov.get();
        a.decomp = decomp.get();
        a.upk = upk.get();
        a.sc = sc.get();
        a.eigScratch = eigScratch.get();
        a.eigLocks = eigLocks.get();
        a.eigSlots = eigSlots;
        return a;
    }

    PropSettings settings() {
        if (settingsDirty) {
            const int nn = n();
            dType.reserve(nn);
            dParam1.reserve(nn);
            dParam2.reserve(nn);
            CUDA_CHECK(cudaMemcpyAsync(dType.get(), type.data(), nn * sizeof(int), cudaMemcpyHostToDevice, stream));
            // SetGaussian keeps sigma^2 in the adaptive proposal (TSimpleMCMC.H:865-866) and sigma
            // itself in TProposeVAATStep (TProposeVAATStep.H:132)
            std::vector<double> p1(param1);
            for (int i = 0; i < nn; ++i)
                if (type[i] == 0 && propKind == SMCMC_PROPOSAL_VAAT) p1[i] = gaussSigma[i];
            CUDA_CHECK(cudaMemcpyAsync(dParam1.get(), p1.data(), nn * sizeof(double), cudaMemcpyHostToDevice, stream));
            CUDA_CHECK(cudaMemcpyAsync(dParam2.get(), param2.data(), nn * sizeof(double), cudaMemcpyHostToDevice, stream));
            const size_t nc = corrValue.size();
            if (nc) {
                dCorr1.reserve(nc);
                dCorr2.reserve(nc);
                dCorrValue.reserve(nc);
                CUDA_CHECK(cudaMemcpyAsync(dCorr1.get(), corrDim1.data(), nc * sizeof(int), cudaMemcpyHostToDevice, stream));
                CUDA_CHECK(cudaMemcpyAsync(dCorr2.get(), corrDim2.data(), nc * sizeof(int), cudaMemcpyHostToDevice, stream));
                CUDA_CHECK(cudaMemcpyAsync(dCorrValue.get(), corrValue.data(), nc * sizeof(double), cudaMemcpyHostToDevice, stream));
            }
            // the host vectors may change before the copies run
            CUDA_CHECK(cudaStreamSynchronize(stream));
            settingsDirty = false;
        }
        PropSettings ps;
        ps.n = n();
        ps.tri = tri();
        ps.covStride = covStride;
        ps.upkStride = upkStride;
        ps.ijTab = ijTab.get();
        ps.covFrozen = covFrozen;
        ps.stepRMSWindow = stepRMSWindow;
        ps.ncorr = (int)corrValue.size();
        ps.anyUniform = 0;
        for (int t : type) ps.anyUniform |= (t == 1);
        ps.covWindow = covWindow;
        ps.accWindow = accWindow;
        ps.target = target;
        ps.covDeweight = covDeweight;
        ps.accDeweight = accDeweight;
        ps.maxCorr = maxCorr;
        ps.type = dType.get();
        ps.param1 = dParam1.get();
        ps.param2 = dParam2.get();
        ps.corrDim1 = dCorr1.get();
        ps.corrDim2 = dCorr2.get();
        ps.corrValue = dCorrValue.get();
        return ps;
    }

    // The n-dependent defaults of InitializeState (TSimpleMCMC.H:1693-1711).
    void resolveInitDefaults() {
        const int nn = n();
        if (accWindow < 0) accWindow = std::pow(1.0 * nn, 1.5) + 1000;     // :1693-1695
        if (target < 1E-4) target = (nn > 4) ? 0.234 : 0.44;               // :1699-1711
    }
    // ... and of ResetProposal (:1468-1480).
    void resolveResetDefaults() {
        const int nn = n();
        int minWindow = 100 + 4 * nn;
        if (covWindow < minWindow) {
            covWindow = nn;
            covWindow *= nn;
            covWindow *= nn;
            covWindow += minWindow;
            double r = std::numeric_limits<double>::epsilon();
            covWindow = std::min(covWindow, std::sqrt(1.0 / r));
        }
        if (target < 0.0) throw Error(SMCMC_ERR_RUNTIME, "Target acceptance not initialized");
    }

    // ---- likelihood evaluation on device arrays ----------------------------
    void evaluate(const double* xDev, int m, double* llhDev, double* histDev) {
        switch (cfg.likelihood) {
        case SMCMC_LLH_FAKE:
        case SMCMC_LLH_FAKE2:
            evaluateFake(xDev, m, llhDev, histDev);
            break;
        case SMCMC_LLH_UNBINNED:
            evaluateUnbinned(xDev, m, llhDev);
            break;
        case SMCMC_LLH_USER: {
            // the user's functor: its kernel lives in the user's translation unit
            if (!userOps.likelihood) throw Error(SMCMC_ERR_LOGIC, "user functor not registered (smcmc_user_set_ops)");
            const int rc = userOps.likelihood(userOps.ctx, xDev, m, n(), llhDev, (void*)stream);
            if (rc != 0) throw Error(SMCMC_ERR_CUDA, std::string("user likelihood launch failed: ") +
                                                     cudaGetErrorString((cudaError_t)rc));
            launched();
            break;
        }
        case SMCMC_LLH_DUMMY: {
            if (errDim != n()) throw Error(SMCMC_ERR_LOGIC, "error matrix not set (smcmc_dummy_set_error)");
            if (dummyMode == SMCMC_DUMMY_TENSOR) {
                // L = -1/2 x . (Error^T x): the contraction on the FP64 tensor cores
                dim3 grid(ceilDiv(n(), kDmmaBN), ceilDiv(m, kDmmaBM));
                dummyPartials.reserve((size_t)m * grid.x);
                launchDummyContractDmma(stream, xDev, errMatrixT.get(), dummyPartials.get(), nullptr, 0, m, n(), 1);
                launched();
                kDummyLlhFromPartials<<<ceilDiv(m, 128), 128, 0, stream>>>(dummyPartials.get(), (int)grid.x, m, llhDev);
                launched();
                break;
            }
            // points per block: as many warps as fit the shared-memory tile, one
            // warp when there are too few points to fill the SMs otherwise
            int warps = (int)std::min<size_t>(4, ((200u << 10) - 2 * ((size_t)n() + 1) * 8) / ((size_t)n() * 8 * 32));
            if (warps >= 1) {
                if (m <= smCount * 32 * 2) warps = 1;
                const int width = warps * 32;
                const size_t smem = ((size_t)n() * width + 2 * (((size_t)n() + 1) & ~(size_t)1)) * sizeof(double);
                if (smem > dummySmemSet) {
                    CUDA_CHECK(cudaFuncSetAttribute(kDummyLikelihood, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                    dummySmemSet = smem;
                }
                kDummyLikelihood<<<ceilDiv(m, width), width, smem, stream>>>(xDev, m, n(), errMatrixT.get(), llhDev);
                launched();
                break;
            }
            // dimension too large for the tile: the generic kernel
            kSimpleLikelihood<<<ceilDiv(m, 128), 128, 0, stream>>>(cfg.likelihood, xDev, m, n(), errMatrix.get(), llhDev);
            launched();
            break;
        }
        default:
            kSimpleLikelihood<<<ceilDiv(m, 128), 128, 0, stream>>>(cfg.likelihood, xDev, m, n(),
                                                                  errMatrix.get(), llhDev);
            launched();
        }
    }

    PairLaunch pairLaunch(int m, int stride) {
        PairLaunch L;
        L.events = fakeEvents.get();
        L.filterTiles = fakeFilterTiles.get();
        // Work items = (chunk of one class) x (tile of 256 points).  Pick the
        // chunk length so that the grid is close to a whole number of waves of
        // (SMs x resident CTAs): equal-cost items, no ragged last wave.
        const int pointTiles = ceilDiv(m, kPairThreads);
        int64_t total = 0;
        for (int c = 0; c < kFakeClasses; ++c) total += fakeClassCount[c];
        const int64_t slots = (int64_t)smCount * kPairCtasPerSm;
        int64_t waves = (total * pointTiles + slots * kPairChunk - 1) / (slots * kPairChunk);
        if (waves < 1) waves = 1;
        int64_t chunkEvents = (total * pointTiles + slots * waves - 1) / (slots * waves);
        chunkEvents = (chunkEvents + kPairTile - 1) / kPairTile * kPairTile;
        if (chunkEvents < kPairTile) chunkEvents = kPairTile;
        // the per-class round-up can spill a few items into one more wave:
        // lengthen the chunk until the grid fits in `waves` waves
        auto items = [&](int64_t ce) {
            int64_t n = 0;
            for (int c = 0; c < kFakeClasses; ++c) n += (fakeClassCount[c] + ce - 1) / ce;
            return n * pointTiles;
        };
        while (chunkEvents < kPairChunk && items(chunkEvents) > slots * waves) chunkEvents += kPairTile;
        if (chunkEvents > kPairChunk) chunkEvents = kPairChunk;
        L.chunkEvents = (int)chunkEvents;
        int chunks = 0;
        for (int c = 0; c < kFakeClasses; ++c) {
            L.classBase[c] = fakeClassBase[c];
            L.classCount[c] = fakeClassCount[c];
            L.classReal[c] = fakeClassReal[c];
            for (int b = 0; b < kMassBands; ++b) L.bandStart[c][b] = fakeBandStart[c][b];
            L.chunkBase[c] = chunks;
            chunks += (int)((fakeClassCount[c] + chunkEvents - 1) / chunkEvents);
        }
        L.chunkBase[kFakeClasses] = chunks;
        L.skipTiles = noTileSkip ? 0 : 1;
        L.chains = fakeChains.get();
        L.filterChains = fakeFilterChains.get();
        L.numPoints = m;
        L.pointStride = stride;
        L.blockPoints = fakeBlockPoints > 0 ? fakeBlockPoints : stride;
        L.counts = fakeCounts.get();
        L.stats = collectStats ? fakeStats.get() : nullptr;
        return L;
    }
    bool collectStats = false;
    size_t dummySmemSet = 48 << 10;
    size_t gramSmemSet = 0;
    // event-sharded evaluation: the count table in blocks of this many points (one block per
    // rank of the event group), 0 = one block
    int fakeBlockPoints = 0;
    bool wantFullCounts = false;                    // the caller reads the whole count table back
    DeviceBuffer<uint32_t> fakeCountsMine;          // the block this rank finishes
    DeviceBuffer<double> fakeLlhGather;
    int eventRank() const { return worldRank % eventGroup; }

    void evaluateFake(const double* xDev, int m, double* llhDev, double* histDev) {
        if (fakeEventCount < 0) throw Error(SMCMC_ERR_LOGIC, "events not set (smcmc_fake_set_events)");
        if (!fakeDataSet) throw Error(SMCMC_ERR_LOGIC, "data histograms not set (smcmc_fake_set_data)");
        int stride = (m + 31) / 32 * 32;
        // Events split over the G ranks of an event group: every rank counts its events for
        // ALL points, then the table is reduce-scattered over points -- rank r receives the
        // summed block r, turns it into log-likelihoods (1/G of the finish work) and the
        // values are all-gathered.  Half the bytes of an all-reduce of the table, and integer
        // sums: the result does not depend on the split.  (Few points, or a caller that wants
        // the histograms / the whole table: one block, all-reduce.)
        const int G = eventGroup;
        const bool scatter = eventComm && G > 1 && !histDev && !wantFullCounts && m >= kPairThreads * G;
        fakeBlockPoints = 0;
        if (scatter) {
            fakeBlockPoints = ceilDiv(ceilDiv(m, G), kPairThreads) * kPairThreads;
            stride = fakeBlockPoints * G;
        }
        fakeChains.reserve(stride);
        fakeFilterChains.reserve(stride);
        fakeCounts.reserve((size_t)kFakeSlots * stride);
        fakeCountStride = stride;
        const bool streaming = m <= kStreamMaxChains && !std::getenv("SMCMC_FAKE_NO_STREAM");
        // few points: the (small) count table is cleared by the prepare kernel, no memset node
        if (!streaming) CUDA_CHECK(cudaMemsetAsync(fakeCounts.get(), 0, (size_t)kFakeSlots * stride * sizeof(uint32_t), stream));
        kFakePrepareChains<<<ceilDiv(m, 128), 128, 0, stream>>>(xDev, m, n(), fakeExposure, fakeChains.get(),
                                                                fakeFilterChains.get(), exactOnly ? 1 : 0,
                                                                cfg.likelihood == SMCMC_LLH_FAKE2 ? 1 : 0,
                                                                streaming ? fakeCounts.get() : nullptr,
                                                                streaming ? kFakeSlots * stride : 0,
                                                                fakeIrregular.get(), streaming ? fakeIrregularCount : 0, stride);
        launched();

        PairLaunch L = pairLaunch(m, stride);
        const int chunks = L.chunkBase[kFakeClasses];
        if (chunks > 0) {
            const int pointTiles = ceilDiv(m, kPairThreads);
            cudaEvent_t e0 = nullptr, e1 = nullptr;
            if (timing) {
                CUDA_CHECK(cudaEventCreate(&e0));
                CUDA_CHECK(cudaEventCreate(&e1));
                CUDA_CHECK(cudaEventRecord(e0, stream));
            }
            if (streaming) {
                // few chains: events streamed once, chains looped per event (fake_likelihood.cuh)
                int64_t tiles = 0;
                for (int c = 0; c < kFakeClasses; ++c) tiles += fakeClassCount[c] / kPairTile;
                const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)smCount * 8, (tiles + 7) / 8));
                if (std::getenv("SMCMC_STREAM_PREFETCH")) kFakeStream<true><<<blocks, kStreamThreads, 0, stream>>>(L);
                else kFakeStream<false><<<blocks, kStreamThreads, 0, stream>>>(L);
            } else
                kFakePairs<<<(unsigned)chunks * (unsigned)pointTiles, kPairThreads, kPairSmemBytes, stream>>>(L);
            launched();
            if (timing) {
                CUDA_CHECK(cudaEventRecord(e1, stream));
                pairEvents.emplace_back(e0, e1);
            }
            ++pairLaunches;
        }
        if (fakeIrregularCount > 0 && !streaming) {                       // (few points: kFakePrepareChains took them along)
            long long pairs = (long long)fakeIrregularCount * m;
            kFakePairsGeneric<<<ceilDiv(pairs, 256), 256, 0, stream>>>(fakeIrregular.get(), fakeIrregularCount,
                                                                       xDev, m, n(), fakeCounts.get(), L.blockPoints);
            launched();
        }
        if (scatter) {
            NcclApi& nccl = NcclApi::get();
            const int per = fakeBlockPoints, r = eventRank();
            const size_t blockWords = (size_t)kFakeSlots * per;
            fakeCountsMine.reserve(blockWords);
            fakeLlhGather.reserve((size_t)per * G);
            nccl.check(nccl.ReduceScatter(fakeCounts.get(), fakeCountsMine.get(), blockWords, ncclUint32, ncclSum, eventComm,
                                          stream), "reduce-scatter of event counts");
            const int first = r * per, mine = std::max(0, std::min(per, m - first));
            if (mine > 0) {
                if (cfg.likelihood == SMCMC_LLH_FAKE2)
                    kFake2Finish<<<ceilDiv(mine, 32), 32 * kFinishWarps, kFinish2SmemBytes, stream>>>(
                        fakeCountsMine.get(), per, mine, fakeChains.get() + first, fakeData.get(),
                        xDev + (size_t)first * n(), n(), fakeLlhGather.get() + first, nullptr);
                else
                    finishFake(fakeCountsMine.get(), per, mine, fakeChains.get() + first, fakeLlhGather.get() + first, nullptr);
                launched();
            }
            nccl.check(nccl.AllGather(fakeLlhGather.get() + first, fakeLlhGather.get(), (size_t)per, ncclDouble, eventComm,
                                      stream), "all-gather of log-likelihoods");
            CUDA_CHECK(cudaMemcpyAsync(llhDev, fakeLlhGather.get(), (size_t)m * sizeof(double), cudaMemcpyDeviceToDevice, stream));
            return;
        }
        if (eventComm) {
            // events are split over the ranks of the event group: the integer
            // counts add exactly, so the result does not depend on the split
            NcclApi& nccl = NcclApi::get();
            nccl.check(nccl.AllReduce(fakeCounts.get(), fakeCounts.get(), (size_t)kFakeSlots * stride, ncclUint32,
                                      ncclSum, eventComm, stream), "all-reduce of event counts");
        }
        if (cfg.likelihood == SMCMC_LLH_FAKE2)
            kFake2Finish<<<ceilDiv(m, 32), 32 * kFinishWarps, kFinish2SmemBytes, stream>>>(
                fakeCounts.get(), stride, m, fakeChains.get(), fakeData.get(), xDev, n(), llhDev, histDev);
        else
            finishFake(fakeCounts.get(), stride, m, fakeChains.get(), llhDev, histDev);
        launched();
    }
    // counts -> bin contents -> log-likelihood of m points (kFakeFinish)
    void finishFake(const uint32_t* counts, int stride, int m, const FakeChainParams* chains, double* llhDev, double* histDev) {
        // few points: the bins of a point group are split over kFinishGroups CTAs
        const int pointGroups = ceilDiv(m, kFinishPoints);
        const bool split = pointGroups * 2 <= smCount;
        if (split) {
            fakeTerms.reserve((size_t)m * 150);
            if ((size_t)pointGroups > fakeTickets.count()) {
                fakeTickets.reserve(smCount);
                CUDA_CHECK(cudaMemsetAsync(fakeTickets.get(), 0, fakeTickets.bytes(), stream));
            }
        }
        kFakeFinish<<<dim3(pointGroups, split ? kFinishGroups : 1), 32 * kFinishBinWarps, 0, stream>>>(
            counts, stride, m, chains, fakeData.get(), llhDev, histDev,
            split ? fakeTerms.get() : nullptr, split ? fakeTickets.get() : nullptr);
    }

    void evaluateUnbinned(const double* xDev, int m, double* llhDev) {
        if (unbEventCount < 0) throw Error(SMCMC_ERR_LOGIC, "events not set (smcmc_unbinned_set_events)");
        const int stride = (m + 31) / 32 * 32;
        unbChains.reserve(stride);
        kUnbinnedPrepareChains<<<ceilDiv(m, 128), 128, 0, stream>>>(xDev, m, n(), unbChains.get());
        launched();
        UnbinnedLaunch L;
        L.events = unbEvents.get();
        const int pointTiles = ceilDiv(m, kUnbThreads);
        const int64_t total = unbClassCount[0] + unbClassCount[1];
        // chunk length: about four waves of (SMs x 8 resident CTAs), at most kUnbMaxChunk events
        const int64_t slots = (int64_t)smCount * 8;
        int64_t waves = std::max<int64_t>(1, (total * pointTiles + slots * kUnbMaxChunk - 1) / (slots * kUnbMaxChunk));
        waves = std::max<int64_t>(waves, std::min<int64_t>(4, (total * pointTiles) / (slots * kUnbTile) + 1));
        int64_t chunkEvents = (total * pointTiles + slots * waves - 1) / (slots * waves);
        chunkEvents = std::min<int64_t>(kUnbMaxChunk, std::max<int64_t>(kUnbTile, (chunkEvents + kUnbTile - 1) / kUnbTile * kUnbTile));
        L.chunkEvents = (int)chunkEvents;
        int chunks = 0;
        for (int c = 0; c < 2; ++c) {
            L.classBase[c] = c == 0 ? 0 : unbClassCount[0];
            L.classCount[c] = unbClassCount[c];
            L.chunkBase[c] = chunks;
            chunks += (int)((unbClassCount[c] + chunkEvents - 1) / chunkEvents);
        }
        L.chunkBase[2] = chunks;
        L.chains = unbChains.get();
        L.numPoints = m;
        L.stride = stride;
        unbPartial.reserve((size_t)std::max(chunks, 1) * stride);
        L.partial = unbPartial.get();
        if (chunks > 0) {
            kUnbinnedPairs<<<(unsigned)chunks * (unsigned)pointTiles, kUnbThreads, 0, stream>>>(L);
            launched();
        }
        kUnbinnedFinish<<<ceilDiv(m, 128), 128, 0, stream>>>(unbPartial.get(), chunks, stride, m, llhDev);
        launched();
        if (eventComm) {
            // events are split over the ranks of the event group: the partial
            // log-likelihoods add (the likelihood is a sum over events)
            NcclApi& nccl = NcclApi::get();
            nccl.check(nccl.AllReduce(llhDev, llhDev, (size_t)m, ncclDouble, ncclSum, eventComm, stream),
                       "all-reduce of partial log-likelihoods");
        }
    }

    void collectPairTimings() {
        for (auto& pr : pairEvents) {
            CUDA_CHECK(cudaEventSynchronize(pr.second));
            float ms = 0.f;
            CUDA_CHECK(cudaEventElapsedTime(&ms, pr.first, pr.second));
            pairMs += ms;
            cudaEventDestroy(pr.first);
            cudaEventDestroy(pr.second);
        }
        pairEvents.clear();
    }

    void checkChainStatus() {
        // surfaces what the reference would have thrown inside Step()
        std::vector<ChainScalars> h(E());
        CUDA_CHECK(cudaMemcpyAsync(h.data(), sc.get(), sizeof(ChainScalars) * E(), cudaMemcpyDeviceToHost, stream));
        CUDA_CHECK(cudaStreamSynchronize(stream));
        for (int c = 0; c < E(); ++c) {
            if (h[c].status != 0) {
                throw Error(h[c].status, "chain " + std::to_string(c) +
                                             ": proposal update failed (invalid covariance trace or "
                                             "decomposition of user correlations failed)");
            }
        }
    }

    void stepOnce(int metropolis, const TraceDev& tr, int traceStep) {
        PropSettings ps = settings();
        ChainArrays a = arrays();
        const int blocks = ceilDiv(E(), kWarpsPerBlock);
        const size_t smem = (size_t)kWarpsPerBlock * 3 * n() * sizeof(double);
        if (debugStep()) {
            // forced or scan step (:671-704): no UpdateState, the accept draw is the next
            // gRandom call of the step (slot 0 after a forced point, 1 after the scan draw)
            const bool forced = forcedPending;
            kProposeDebug<<<ceilDiv(E(), 128), 128, 0, stream>>>(a, ps, E(), forced ? forcedStep.get() : nullptr, scanDim,
                                                                 cfg.seed, cfg.chain_offset, stepRef());
            launched();
            forcedPending = false;                                       // fForcedStep.clear(), :677
            vaatSynced = false;
            evaluate(xProp.get(), E(), llhProp.get(), nullptr);
            kAccept<<<ceilDiv(E(), acceptThreads()), acceptThreads(), 0, stream>>>(a, ps, E(), llhProp.get(), cfg.seed,
                                                                                 cfg.chain_offset, stepRef(), metropolis, tr,
                                                                                 traceStep, nullptr, forced ? 0 : 1);
            launched();
            ++stepIndex;
            if (diagOn) diagAccumulate();
            return;
        }
        if (pooledEvery > 0 && usePooledTensor()) {
            // x' = x + (sigma z) . U for all chains as one GEMM on the FP64 tensor cores
            poolZ.reserve((size_t)E() * n());
            poolY.reserve((size_t)E() * n());
            kProposePooled<<<blocks, kWarpsPerBlock * 32, smem, stream>>>(a, ps, pooled(), E(), cfg.seed,
                                                                          cfg.chain_offset, stepRef(), poolZ.get());
            launched();
            launchDummyContractDmma(stream, poolZ.get(), poolDecompT.get(), poolY.get(), nullptr, 0, E(), n(), 0);
            launched();
            kProposePooledFinish<<<blocks, kWarpsPerBlock * 32, (size_t)kWarpsPerBlock * n() * sizeof(double), stream>>>(
                a, ps, E(), poolY.get());
        } else if (pooledEvery > 0 && usePooledTile())
            kProposePooledTile<<<ceilDiv(E(), kPooledTileChains), kPooledTileThreads, pooledTileSmem(n()), stream>>>(
                a, ps, pooled(), E(), cfg.seed, cfg.chain_offset, stepRef());
        else if (pooledEvery > 0)
            kProposePooled<<<blocks, kWarpsPerBlock * 32, smem, stream>>>(a, ps, pooled(), E(), cfg.seed,
                                                                          cfg.chain_offset, stepRef(), nullptr);
        else if (propKind == SMCMC_PROPOSAL_VAAT) {
            if (!vaatSynced) {   // :52 -- once; afterwards kVaatPropose restores the one coordinate that moved
                CUDA_CHECK(cudaMemcpyAsync(xProp.get(), xAcc.get(), sizeof(double) * E() * n(), cudaMemcpyDeviceToDevice, stream));
                vaatSynced = true;
            }
            kVaatPropose<<<ceilDiv(E(), 128), 128, 0, stream>>>(a, vaatArrays(), ps, E(), cfg.seed, cfg.chain_offset, stepRef());
        } else if (staged)
            kProposeStaged<<<E(), kStagedThreads, stagedChainBytes(n(), covStride, upkStride), stream>>>(
                a, ps, E(), cfg.seed, cfg.chain_offset, stepRef());
        else
            kPropose<<<blocks, kWarpsPerBlock * 32, smem, stream>>>(a, ps, E(), cfg.seed, cfg.chain_offset, stepRef());
        launched();
        const int* acceptSlot = propKind == SMCMC_PROPOSAL_VAAT ? (const int*)vState.get() : nullptr;
        if (traceStep < 0 && acceptLocal()) {
            // chain-local likelihood, no trace: likelihood + Metropolis rule in one launch (accept_local.cuh)
            kAcceptLocal<<<ceilDiv(E(), 32 * kAcceptLocalWarps), 32 * kAcceptLocalWarps, acceptLocalSmem(n()), stream>>>(
                a, ps, E(), cfg.likelihood, cfg.seed, cfg.chain_offset, stepRef(), metropolis, acceptSlot);
        } else {
            evaluate(xProp.get(), E(), llhProp.get(), nullptr);
            kAccept<<<ceilDiv(E(), acceptThreads()), acceptThreads(), 0, stream>>>(a, ps, E(), llhProp.get(), cfg.seed,
                                                                                 cfg.chain_offset, stepRef(), metropolis, tr,
                                                                                 traceStep, acceptSlot);
        }
        launched();
        if (graphMode) {
            kBumpStep<<<1, 1, 0, stream>>>(dStep.get());
            launched();
        }
        ++stepIndex;
        if (diagOn) diagAccumulate();
        if (pooledEvery > 0) {
            poolAccumulate(poolStats.get());
            if (stepIndex % (uint32_t)pooledEvery == 0) poolExchange();
        }
    }

    // nsteps Metropolis steps without a trace.  A step is 3 to 8 small launches; for
    // small ensembles the host launch path, not the GPU, sets the pace.  When nothing in
    // the step needs the host (no exchange, no timing, no diagnostics) the loop is
    // captured ONCE as a CUDA graph -- after a plain first step that sizes every buffer --
    // and replayed; the kernels read the step counter from a device word that the graph's
    // last node increments.  Opt-in (SMCMC_GRAPH=1): measured on B200 it gains 2-5 % for
    // 8-256 chains x 4M events and LOSES for one chain (gpurun_out/mid_ensemble.txt);
    // the launch-bound chain-local case is served by kStepsResident instead.
    static constexpr int kGraphMinSteps = 8;
    // kAccept: one thread per chain decides, the warp then copies the rows of its chains that accepted.
    // With few chains per SM the copies of 128-thread blocks leave most SMs idle: one warp per block then.
    int acceptThreads() const { return E() < 2 * smCount * kAcceptThreads ? 32 : kAcceptThreads; }
    bool debugStep() const { return propKind == SMCMC_PROPOSAL_ADAPTIVE && (forcedPending || scanDim >= 0); }
    bool graphable() const {
        const char* g = std::getenv("SMCMC_GRAPH");
        return g && g[0] == '1' && pooledEvery == 0 && !eventComm && !timing && !diagOn && !debugStep();
    }
    // kAcceptLocal instead of likelihood kernel + kAccept (SMCMC_NO_ACCEPT_LOCAL=1: the two launches)
    bool acceptLocalReady = false;
    bool acceptLocal() {
        switch (cfg.likelihood) {
        case SMCMC_LLH_UNIT_GAUSS:
        case SMCMC_LLH_HORRIFIC:
        case SMCMC_LLH_ASYM:
        case SMCMC_LLH_HARD:
            break;
        default:
            return false;
        }
        if (timing || acceptLocalSmem(n()) > 160u * 1024u || std::getenv("SMCMC_NO_ACCEPT_LOCAL")) return false;
        if (!acceptLocalReady) {
            CUDA_CHECK(cudaFuncSetAttribute(kAcceptLocal, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)acceptLocalSmem(n())));
            acceptLocalReady = true;
        }
        return true;
    }
    // The likelihood needs only the chain's own point and the proposal is the per-chain
    // adaptive one: all nsteps steps run in ONE launch with the chain's state resident in
    // shared memory (proposal_resident.cuh).  SMCMC_NO_RESIDENT=1 keeps the three-launch step.
    bool residentable() const {
        if (!resident || pooledEvery > 0 || propKind != SMCMC_PROPOSAL_ADAPTIVE || timing || diagOn || debugStep()) return false;
        if (std::getenv("SMCMC_NO_RESIDENT")) return false;
        // up to one wave of CTAs; a larger ensemble is served as well by the three-launch
        // step (measured, proposal_resident.cuh).  SMCMC_RESIDENT=1 lifts the limit.
        if (E() > residentPerSm * smCount && !std::getenv("SMCMC_RESIDENT")) return false;
        switch (cfg.likelihood) {
        case SMCMC_LLH_UNIT_GAUSS:
        case SMCMC_LLH_HORRIFIC:
        case SMCMC_LLH_ASYM:
        case SMCMC_LLH_HARD:
            return true;
        case SMCMC_LLH_DUMMY:
            // the n^2 ordered terms are summed by one warp here: beyond n = 20 the tiled
            // kDummyLikelihood of the three-launch step is faster (n = 100: 213 vs 461 us per step)
            return dummyMode != SMCMC_DUMMY_TENSOR && errDim == n() && n() <= 20;
        default:
            return false;
        }
    }
    void stepMany(int nsteps, int metropolis) {
        TraceDev none = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
        int done = 0;
        if (forcedPending && nsteps > 0) {            // the forced point is the proposal of the first step only
            stepOnce(metropolis, none, -1);
            done = 1;
            if (nsteps == 1) return;
        }
        if (nsteps - done >= 2 && residentable()) {
            PropSettings ps = settings();
            ChainArrays a = arrays();
            const double* errT = cfg.likelihood == SMCMC_LLH_DUMMY ? errMatrixT.get() : nullptr;
            kStepsResident<<<E(), kStagedThreads, residentChainBytes(n(), covStride, upkStride), stream>>>(
                a, ps, E(), cfg.seed, cfg.chain_offset, stepIndex, nsteps - done, metropolis, cfg.likelihood, errT);
            launched();
            ++residentLaunches;
            stepIndex += (uint32_t)(nsteps - done);
            return;
        }
        if (nsteps - done >= kGraphMinSteps && graphable()) {
            stepOnce(metropolis, none, -1);           // sizes the buffers, uploads dirty settings
            ++done;
            if (!graphStream) {
                CUDA_CHECK(cudaStreamCreateWithFlags(&graphStream, cudaStreamNonBlocking));
                CUDA_CHECK(cudaEventCreateWithFlags(&graphEvent, cudaEventDisableTiming));
            }
            dStep.reserve(1);
            cudaStream_t user = stream;
            kSetStep<<<1, 1, 0, user>>>(dStep.get(), stepIndex);
            CUDA_CHECK(cudaEventRecord(graphEvent, user));
            CUDA_CHECK(cudaStreamWaitEvent(graphStream, graphEvent, 0));
            cudaGraph_t graph = nullptr;
            const int64_t launchesBefore = launches;
            const uint32_t stepBefore = stepIndex;
            bool captured = false;
            stream = graphStream;
            graphMode = true;
            if (cudaStreamBeginCapture(graphStream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                try {
                    stepOnce(metropolis, none, -1);
                    captured = cudaStreamEndCapture(graphStream, &graph) == cudaSuccess && graph != nullptr;
                } catch (...) {
                    cudaStreamEndCapture(graphStream, &graph);
                    captured = false;
                }
            }
            graphMode = false;
            stream = user;
            stepIndex = stepBefore;                   // the captured step has not run
            const int64_t nodes = launches - launchesBefore;
            launches = launchesBefore;
            // the executable graph is kept between calls: a fresh capture of the same
            // topology only updates its node parameters (settings, pointers), which is
            // much cheaper than instantiating it again
            if (captured && graphExec) {
                cudaGraphExecUpdateResultInfo info;
                if (cudaGraphExecUpdate(graphExec, graph, &info) != cudaSuccess) {
                    cudaGetLastError();
                    cudaGraphExecDestroy(graphExec);
                    graphExec = nullptr;
                }
            }
            if (captured && !graphExec && cudaGraphInstantiate(&graphExec, graph, 0) != cudaSuccess) {
                cudaGetLastError();
                graphExec = nullptr;
            }
            if (captured && graphExec) {
                for (; done < nsteps; ++done) {
                    CUDA_CHECK(cudaGraphLaunch(graphExec, graphStream));
                    ++stepIndex;
                    launches += nodes;
                }
                CUDA_CHECK(cudaEventRecord(graphEvent, graphStream));
                CUDA_CHECK(cudaStreamWaitEvent(user, graphEvent, 0));
            } else {
                cudaGetLastError();                   // capture is an optimisation: fall through to the plain loop
            }
            if (graph) cudaGraphDestroy(graph);
        }
        for (; done < nsteps; ++done) stepOnce(metropolis, none, -1);
    }
};

namespace {

template <class F>
int guarded(smcmc_engine* e, F f) {
    try {
        // every entry point works on the engine's device whatever the caller's current one is
        // (allocations come from that device's pool, launches go to a stream of that device)
        if (e) CUDA_CHECK(cudaSetDevice(e->cfg.device));
        f();
        return SMCMC_OK;
    } catch (const Error& err) {
        if (e) e->lastError = err.what();
        else gCreateError = err.what();
        return err.status;
    } catch (const std::exception& err) {
        if (e) e->lastError = err.what();
        else gCreateError = err.what();
        return SMCMC_ERR_RUNTIME;
    }
}

void requireStarted(smcmc_engine* e) {
    if (!e->started) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "Uninitialized starting point");   // TSimpleMCMC.H:371-374
}

}  // namespace

extern "C" {

int smcmc_abi_version(void) { return SMCMC_B200_ABI_VERSION; }

const char* smcmc_last_error(const smcmc_engine* e) {
    return e ? e->lastError.c_str() : gCreateError.c_str();
}

int smcmc_create(const smcmc_config* cfg, smcmc_engine** out) {
    if (out) *out = nullptr;
    smcmc_engine* e = nullptr;
    int rc = guarded(nullptr, [&]() {
        if (!cfg || !out) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null argument");
        if (cfg->struct_size != sizeof(smcmc_config)) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "smcmc_config size mismatch");
        if (cfg->dim < 1 || cfg->chains < 1) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "dim and chains must be positive");
        if (cfg->likelihood < SMCMC_LLH_UNIT_GAUSS || cfg->likelihood > SMCMC_LLH_USER)
            throw Error(SMCMC_ERR_INVALID_ARGUMENT, "unknown likelihood");
        if (cfg->likelihood == SMCMC_LLH_HARD && cfg->dim < 2)
            throw Error(SMCMC_ERR_INVALID_ARGUMENT, "THardLogLikelihood needs two or more dimensions");
        if ((cfg->likelihood == SMCMC_LLH_FAKE || cfg->likelihood == SMCMC_LLH_FAKE2 ||
             cfg->likelihood == SMCMC_LLH_UNBINNED) && cfg->dim != 9)
            throw Error(SMCMC_ERR_INVALID_ARGUMENT, "the event likelihood functors have 9 parameters");
        int count = 0;
        cudaError_t ce = cudaGetDeviceCount(&count);
        if (ce != cudaSuccess || count < 1) {
            cudaGetLastError();
            throw Error(SMCMC_ERR_NO_DEVICE, "no CUDA device: libsmcmc_b200 has no CPU fallback");
        }
        if (cfg->device < 0 || cfg->device >= count) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "bad device ordinal");
        CUDA_CHECK(cudaSetDevice(cfg->device));
        cudaDeviceProp prop;
        CUDA_CHECK(cudaGetDeviceProperties(&prop, cfg->device));
        if (prop.major < 10) throw Error(SMCMC_ERR_NO_DEVICE, "libsmcmc_b200 is built for sm_100a only");

        e = new smcmc_engine;
        e->cfg = *cfg;
        e->smCount = prop.multiProcessorCount;
        const size_t E = cfg->chains, n = cfg->dim;
        e->type.assign(n, 0);
        e->param1.assign(n, 0.0);
        e->param2.assign(n, 0.0);
        e->gaussSigma.assign(n, 0.0);
        e->xAcc.reserve(E * n);
        e->xProp.reserve(E * n);
        e->lastPoint.reserve(E * n);
        e->center.reserve(E * n);
        const size_t tri = n * (n + 1) / 2;
        e->covStride = (int)((tri + 15) / 16 * 16);
        e->upkStride = (upkTotal((int)n) + 15) / 16 * 16;
        e->cov.reserve(E * e->covStride);
        e->decomp.reserve(E * n * n);
        e->upk.reserve(E * e->upkStride);
        {
            std::vector<uint32_t> tab(tri);
            for (size_t i = 0, k = 0; i < n; ++i)
                for (size_t j = 0; j <= i; ++j) tab[k++] = (uint32_t)(i * 8) | ((uint32_t)(j * 8) << 16);
            e->ijTab.reserve(tri);
            CUDA_CHECK(cudaMemcpy(e->ijTab.get(), tab.data(), tri * sizeof(uint32_t), cudaMemcpyHostToDevice));
        }
        // kProposeStaged (one CTA per chain) when at least four chains fit an SM (227 KB)
        {
            const size_t cb = stagedChainBytes((int)n, e->covStride, e->upkStride);
            if ((227 * 1024) / (cb + 1024) >= 4 && n < 8192 && !std::getenv("SMCMC_PROPOSE_GENERIC")) {
                e->staged = true;
                CUDA_CHECK(cudaFuncSetAttribute(kProposeStaged, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cb));
            }
            // kStepsResident (whole steps out of shared memory) when one chain fits an SM
            const size_t rb = residentChainBytes((int)n, e->covStride, e->upkStride);
            if (rb <= 200u * 1024u && n < 8192) {
                e->resident = true;
                e->residentPerSm = (int)std::min<size_t>(6, (227 * 1024) / (rb + 1024));
                CUDA_CHECK(cudaFuncSetAttribute(kStepsResident, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rb));
            }
        }
        e->llhProp.reserve(E);
        e->sc.reserve(E);
        e->okDev.reserve(E);
        // scratch pool for the eigen-decomposition fallback: at most 64 slots, <= 256 MB
        e->eigSlots = (int)std::min<size_t>(std::min<size_t>(E, 64), std::max<size_t>(1, (256u << 20) / (2 * n * n * 8)));
        e->eigScratch.reserve((size_t)e->eigSlots * 2 * n * n);
        e->eigLocks.reserve(e->eigSlots);
        CUDA_CHECK(cudaMemset(e->eigLocks.get(), 0, e->eigSlots * sizeof(int)));
        CUDA_CHECK(cudaMemset(e->sc.get(), 0, e->sc.bytes()));
        CUDA_CHECK(cudaMemset(e->cov.get(), 0, e->cov.bytes()));
        CUDA_CHECK(cudaMemset(e->decomp.get(), 0, e->decomp.bytes()));
        CUDA_CHECK(cudaMemset(e->upk.get(), 0, e->upk.bytes()));
        CUDA_CHECK(cudaMemset(e->center.get(), 0, e->center.bytes()));
        CUDA_CHECK(cudaMemset(e->lastPoint.get(), 0, e->lastPoint.bytes()));
        // TProposeAdaptiveStep constructor defaults, TSimpleMCMC.H:642-655
        std::vector<ChainScalars> init(E);
        std::memset(init.data(), 0, sizeof(ChainScalars) * E);
        for (size_t c = 0; c < E; ++c) {
            init[c].rigidity = 2.0;
            init[c].nextUpdate = -1;
        }
        CUDA_CHECK(cudaMemcpy(e->sc.get(), init.data(), sizeof(ChainScalars) * E, cudaMemcpyHostToDevice));
        e->forceGeneric = std::getenv("SMCMC_FAKE_FORCE_GENERIC") != nullptr;
        e->exactOnly = std::getenv("SMCMC_FAKE_EXACT") != nullptr;
        e->noTileSkip = std::getenv("SMCMC_FAKE_NO_SKIP") != nullptr;
        e->fakeStats.reserve(4);
        CUDA_CHECK(cudaMemset(e->fakeStats.get(), 0, 4 * sizeof(unsigned long long)));

        if (cfg->likelihood == SMCMC_LLH_UNBINNED) {
            double consts[4] = {std::tan(M_PI * (0.05 - 0.5)), std::tan(M_PI * (0.5 - 0.5)), M_PI, 0.0};
            CUDA_CHECK(cudaMemcpyToSymbol(gFakeConst, consts, sizeof(consts)));
        }
        if (cfg->likelihood == SMCMC_LLH_FAKE || cfg->likelihood == SMCMC_LLH_FAKE2) {
            CUDA_CHECK(cudaFuncSetAttribute(kFake2Finish, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFinish2SmemBytes));
            // Pre-images of the TH1 bin edges under this host's exp: bin(exp(l)).
            double edges[52];
            edges[0] = -std::numeric_limits<double>::infinity();
            for (int k = 1; k <= 49; ++k) {
                edges[k] = firstLogWhere(
                    [k](double mass) { return 1 + int(50 * (mass - 0.0) / (500.0 - 0.0)) >= k + 1; },
                    std::log(10.0 * k) - 0.01, std::log(10.0 * k) + 0.01);
            }
            // dropped when Mass > 500 (FakeLikelihood.H:203) or in the overflow bin (!(x<500))
            edges[50] = firstLogWhere([](double mass) { return !(mass < 500.0); }, std::log(500.0) - 0.01,
                                      std::log(500.0) + 0.01);
            edges[51] = std::numeric_limits<double>::infinity();
            CUDA_CHECK(cudaMemcpyToSymbol(gEdges, edges, sizeof(edges)));
            double consts[4] = {std::tan(M_PI * (0.05 - 0.5)), std::tan(M_PI * (0.5 - 0.5)), M_PI, 0.0};
            CUDA_CHECK(cudaMemcpyToSymbol(gFakeConst, consts, sizeof(consts)));
            CUDA_CHECK(cudaFuncSetAttribute(kFakePairs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPairSmemBytes));
            e->fakeData.reserve(150);
        }
        if ((size_t)kWarpsPerBlock * 3 * n * sizeof(double) > 48 * 1024) {
            CUDA_CHECK(cudaFuncSetAttribute(kPropose, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)((size_t)kWarpsPerBlock * 3 * n * sizeof(double))));
            CUDA_CHECK(cudaFuncSetAttribute(kProposePooled, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)((size_t)kWarpsPerBlock * 3 * n * sizeof(double))));
        }
        *out = e;
    });
    if (rc != SMCMC_OK && e) delete e;
    return rc;
}

int smcmc_comm_unique_id(char* out, size_t bytes) {
    return guarded(nullptr, [&]() {
        if (!out || bytes < sizeof(ncclUniqueId)) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "need 128 bytes");
        NcclApi& nccl = NcclApi::get();
        ncclUniqueId id;
        nccl.check(nccl.GetUniqueId(&id), "ncclGetUniqueId");
        std::memcpy(out, &id, sizeof id);
    });
}

int smcmc_comm_init(smcmc_engine* e, const char* idBytes, size_t bytes, int world, int rank, int eventGroup) {
    return guarded(e, [&]() {
        if (!idBytes || bytes < sizeof(ncclUniqueId)) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "need the 128-byte unique id");
        if (world < 1 || rank < 0 || rank >= world || eventGroup < 1 || world % eventGroup)
            throw Error(SMCMC_ERR_INVALID_ARGUMENT, "bad world / rank / event group");
        if (e->worldComm) throw Error(SMCMC_ERR_LOGIC, "communicator already initialised");
        NcclApi& nccl = NcclApi::get();
        ncclUniqueId id;
        std::memcpy(&id, idBytes, sizeof id);
        CUDA_CHECK(cudaSetDevice(e->cfg.device));
        nccl.check(nccl.CommInitRank(&e->worldComm, world, id, rank), "ncclCommInitRank");
        e->worldSize = world;
        e->worldRank = rank;
        e->eventGroup = eventGroup;
        if (eventGroup > 1)
            nccl.check(nccl.CommSplit(e->worldComm, rank / eventGroup, rank % eventGroup, &e->eventComm, nullptr),
                       "ncclCommSplit");
    });
}

int smcmc_destroy(smcmc_engine* e) {
    if (!e) return SMCMC_OK;
    cudaSetDevice(e->cfg.device);
    cudaDeviceSynchronize();
    if (e->graphExec) cudaGraphExecDestroy(e->graphExec);
    if (e->graphStream) cudaStreamDestroy(e->graphStream);
    if (e->graphEvent) cudaEventDestroy(e->graphEvent);
    if (e->eventComm) NcclApi::get().CommDestroy(e->eventComm);
    if (e->worldComm) NcclApi::get().CommDestroy(e->worldComm);
    for (auto& pr : e->pairEvents) {
        cudaEventDestroy(pr.first);
        cudaEventDestroy(pr.second);
    }
    delete e;
    return SMCMC_OK;
}

int smcmc_set_stream(smcmc_engine* e, void* s) {
    return guarded(e, [&]() {
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        e->stream = (cudaStream_t)s;
    });
}

int smcmc_sync(smcmc_engine* e) {
    return guarded(e, [&]() {
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        if (e->started) e->checkChainStatus();
    });
}

int smcmc_prop_set(smcmc_engine* e, int field, double v) {
    return guarded(e, [&]() {
        bool perChain = false;
        switch (field) {
        case SMCMC_PROP_SIGMA: perChain = true; break;
        case SMCMC_PROP_TARGET_ACCEPTANCE: e->target = v; break;
        case SMCMC_PROP_ACCEPTANCE_WINDOW:
            e->accWindow = v;
            e->vaatWindow = (int)v;                                            // TProposeVAATStep.H:136 (int member)
            break;
        case SMCMC_PROP_KIND:
            if (e->started) throw Error(SMCMC_ERR_LOGIC, "the proposal kind is chosen before Start()");
            if (v != SMCMC_PROPOSAL_ADAPTIVE && v != SMCMC_PROPOSAL_VAAT)
                throw Error(SMCMC_ERR_INVALID_ARGUMENT, "unknown proposal kind");
            e->propKind = (int)v;
            e->settingsDirty = true;
            break;
        case SMCMC_PROP_ACCEPTANCE_RIGIDITY: perChain = true; break;
        case SMCMC_PROP_ACCEPTANCE_DEWEIGHT: e->accDeweight = v; break;
        case SMCMC_PROP_COVARIANCE_WINDOW: e->covWindow = (int)v; break;      // SetCovarianceWindow(int)
        case SMCMC_PROP_COVARIANCE_DEWEIGHT: e->covDeweight = v; break;
        case SMCMC_PROP_COVARIANCE_FROZEN: e->covFrozen = (v != 0.0); break;
        case SMCMC_PROP_COVARIANCE_TRIALS: perChain = true; break;
        case SMCMC_PROP_CENTER_TRIALS: perChain = true; break;
        case SMCMC_PROP_NEXT_UPDATE: perChain = true; break;
        case SMCMC_PROP_MAX_CORRELATION: e->maxCorr = v; break;
        case SMCMC_PROP_STEP_RMS_WINDOW: e->stepRMSWindow = (int)v; break;
        case SMCMC_PROP_POOLED_TENSOR:
            e->pooledTensor = (v < 0) ? -1 : (v != 0.0);
            if (e->started && e->pooledEvery > 0 && e->poolStats.count() != 0) e->poolTranspose();
            break;
        case SMCMC_PROP_POOLED_EVERY:
            if (v < 0) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "pooled exchange period must be >= 0");
            e->pooledEvery = (int)v;
            if (e->started && e->pooledEvery > 0 && e->poolStats.count() == 0) e->poolInit();
            break;
        default: throw Error(SMCMC_ERR_INVALID_ARGUMENT, "unknown proposal field");
        }
        if (perChain) {
            kSetScalar<<<ceilDiv(e->E(), 128), 128, 0, e->stream>>>(e->sc.get(), e->E(), field, v);
            e->launched();
        }
    });
}

int smcmc_prop_set_gaussian(smcmc_engine* e, int d, double sigma) {
    return guarded(e, [&]() {
        if (d < 0 || d >= e->n()) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "dimension out of range");   // :856-860
        e->type[d] = 0;
        e->param1[d] = sigma * sigma;                                                                  // :865-866
        e->gaussSigma[d] = sigma;
        e->settingsDirty = true;
    });
}

int smcmc_prop_set_uniform(smcmc_engine* e, int d, double lo, double hi) {
    return guarded(e, [&]() {
        if (d < 0 || d >= e->n()) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "dimension out of range");   // :834-839
        e->type[d] = 1;
        e->param1[d] = lo;
        e->param2[d] = hi;
        e->settingsDirty = true;
    });
}

int smcmc_prop_set_correlation(smcmc_engine* e, int d1, int d2, double c) {
    return guarded(e, [&]() {
        if (d1 < 0 || d1 >= e->n() || d2 < 0 || d2 >= e->n())
            throw Error(SMCMC_ERR_INVALID_ARGUMENT, "dimension out of range");
        if (d1 == d2) return;                                                                          // :884-890
        if (c < -e->maxCorr) c = -e->maxCorr;                                                          // :891-902
        if (c > e->maxCorr) c = e->maxCorr;
        e->corrDim1.push_back(d1);
        e->corrDim2.push_back(d2);
        e->corrValue.push_back(c);
        e->settingsDirty = true;
    });
}

int smcmc_prop_reset_correlations(smcmc_engine* e) {
    return guarded(e, [&]() {
        e->corrDim1.clear();
        e->corrDim2.clear();
        e->corrValue.clear();
        e->settingsDirty = true;
    });
}

static void userUpdate(smcmc_engine* e, int reset) {
    requireStarted(e);
    if (e->pooledEvery > 0) {
        // pooled mode: UpdateProposal = exchange + refactor now; ResetProposal
        // additionally forgets the accumulated statistics afterwards
        e->poolExchange();
        if (reset) CUDA_CHECK(cudaMemsetAsync(e->poolStats.get(), 0, e->poolStatCount() * sizeof(double), e->stream));
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        return;
    }
    if (reset) e->resolveResetDefaults();
    PropSettings ps = e->settings();
    kUserUpdate<<<ceilDiv(e->E(), kWarpsPerBlock), kWarpsPerBlock * 32, 0, e->stream>>>(e->arrays(), ps, e->E(), reset);
    e->launched();
    e->checkChainStatus();
}

int smcmc_prop_update(smcmc_engine* e) {
    return guarded(e, [&]() {
        if (e->propKind == SMCMC_PROPOSAL_VAAT)
            throw Error(SMCMC_ERR_LOGIC, "TProposeVAATStep has no UpdateProposal / ResetProposal to call");
        userUpdate(e, 0);
    });
}

int smcmc_prop_reset(smcmc_engine* e) {
    return guarded(e, [&]() {
        if (e->propKind == SMCMC_PROPOSAL_VAAT)
            throw Error(SMCMC_ERR_LOGIC, "TProposeVAATStep has no UpdateProposal / ResetProposal to call");
        userUpdate(e, 1);
    });
}

int smcmc_user_set_ops(smcmc_engine* e, const smcmc_user_ops* ops) {
    return guarded(e, [&]() {
        if (e->cfg.likelihood != SMCMC_LLH_USER) throw Error(SMCMC_ERR_LOGIC, "engine was not created with SMCMC_LLH_USER");
        if (!ops || ops->struct_size != sizeof(smcmc_user_ops) || !ops->likelihood)
            throw Error(SMCMC_ERR_INVALID_ARGUMENT, "bad smcmc_user_ops");
        e->userOps = *ops;
    });
}

int smcmc_prop_force_step(smcmc_engine* e, const double* x, int per_chain) {
    return guarded(e, [&]() {
        if (e->propKind != SMCMC_PROPOSAL_ADAPTIVE) throw Error(SMCMC_ERR_LOGIC, "ForceStep belongs to TProposeAdaptiveStep");
        if (!x) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "Invalid forced step point.");          // :812-814
        const size_t E = e->E(), n = e->n();
        e->forcedStep.reserve(E * n);
        if (per_chain) {
            CUDA_CHECK(cudaMemcpyAsync(e->forcedStep.get(), x, E * n * 8, cudaMemcpyHostToDevice, e->stream));
        } else {
            std::vector<double> all(E * n);
            for (size_t c = 0; c < E; ++c) std::copy(x, x + n, all.begin() + c * n);
            CUDA_CHECK(cudaMemcpyAsync(e->forcedStep.get(), all.data(), E * n * 8, cudaMemcpyHostToDevice, e->stream));
        }
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        e->forcedPending = true;
    });
}

int smcmc_prop_set_scan_dimension(smcmc_engine* e, int dim) {
    return guarded(e, [&]() {
        if (e->propKind != SMCMC_PROPOSAL_ADAPTIVE) throw Error(SMCMC_ERR_LOGIC, "SetScanDimension belongs to TProposeAdaptiveStep");
        e->scanDim = (dim < 0 || dim >= e->n()) ? -1 : dim;                                     // :827-829
    });
}

int smcmc_prop_set_center(smcmc_engine* e, const double* v, int per_chain) {
    return guarded(e, [&]() {
        if (!v) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null centre");
        const size_t E = e->E(), n = e->n();
        DeviceBuffer<double> tmp;
        tmp.reserve(per_chain ? E * n : n);
        CUDA_CHECK(cudaMemcpyAsync(tmp.get(), v, (per_chain ? E * n : n) * 8, cudaMemcpyHostToDevice, e->stream));
        kSetCenter<<<ceilDiv((long long)(E * n), 256), 256, 0, e->stream>>>(e->center.get(), tmp.get(), (int)E, (int)n, per_chain ? 1 : 0);
        e->launched();
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
    });
}

int smcmc_fake_set_events(smcmc_engine* e, const smcmc_event* events, int64_t count) {
    return guarded(e, [&]() {
        if (e->cfg.likelihood != SMCMC_LLH_FAKE && e->cfg.likelihood != SMCMC_LLH_FAKE2)
            throw Error(SMCMC_ERR_LOGIC, "engine was not created with SMCMC_LLH_FAKE or SMCMC_LLH_FAKE2");
        if (count < 0 || (count > 0 && !events)) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "bad event array");
        if (count > 0xffffffffLL) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "more than 2^32 events per engine");
        // One arena for everything that only lives during the re-layout (raw
        // records, sort keys and indices in and out, the sort's scratch, the
        // small counters): one allocation and one release per upload.
        size_t sortBytes = 0;
        if (count > 0)
            CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, sortBytes, (unsigned long long*)nullptr,
                                                       (unsigned long long*)nullptr, (unsigned int*)nullptr,
                                                       (unsigned int*)nullptr, (int)count, 0, kSortKeyBits, e->stream));
        auto align = [](size_t b) { return (b + 255) / 256 * 256; };
        const size_t n = (size_t)count;
        constexpr int kCountSlots = 8 * kBandSlots;            // per (class, mass band), kFakeCountClasses
        const size_t offRaw = 0;
        const size_t offKeysIn = offRaw + align(n * sizeof(smcmc_event));
        const size_t offKeysOut = offKeysIn + align(n * 8);
        const size_t offIndexIn = offKeysOut + align(n * 8);
        const size_t offIndexOut = offIndexIn + align(n * 4);
        const size_t offSort = offIndexOut + align(n * 4);
        const size_t offSmall = offSort + align(sortBytes);
        DeviceBuffer<unsigned char> arena;
        arena.reserve(offSmall + 1024);
        unsigned char* base0 = arena.get();
        smcmc_event* raw = (smcmc_event*)(base0 + offRaw);
        unsigned long long* keysIn = (unsigned long long*)(base0 + offKeysIn);
        unsigned long long* keysOut = (unsigned long long*)(base0 + offKeysOut);
        unsigned int* indexIn = (unsigned int*)(base0 + offIndexIn);
        unsigned int* indexOut = (unsigned int*)(base0 + offIndexOut);
        unsigned long long* counters = (unsigned long long*)(base0 + offSmall);        // 64 x u64
        int64_t* baseDev = (int64_t*)(base0 + offSmall + 512);                           // 8 x i64
        int64_t* startDev = (int64_t*)(base0 + offSmall + 576);                          // 8 x i64
        CUDA_CHECK(cudaMemsetAsync(counters, 0, kCountSlots * sizeof(unsigned long long), e->stream));
        unsigned long long bandCount[kCountSlots] = {0};
        if (count > 0) {
            CUDA_CHECK(cudaMemcpyAsync(raw, events, sizeof(smcmc_event) * count, cudaMemcpyHostToDevice, e->stream));
            kFakeCountClasses<<<ceilDiv(count, 256), 256, 0, e->stream>>>(raw, count, counters, e->forceGeneric);
            e->launched();
            // the keys do not depend on the counts: queue them before the read-back
            kFakeSortKeys<<<ceilDiv(count, 256), 256, 0, e->stream>>>(raw, count, keysIn, indexIn, e->forceGeneric);
            e->launched();
            CUDA_CHECK(cub::DeviceRadixSort::SortPairs(base0 + offSort, sortBytes, keysIn, keysOut, indexIn, indexOut,
                                                       (int)count, 0, kSortKeyBits, e->stream));
            e->launched();
            CUDA_CHECK(cudaMemcpyAsync(bandCount, counters, sizeof(bandCount), cudaMemcpyDeviceToHost, e->stream));
            CUDA_CHECK(cudaStreamSynchronize(e->stream));
        }
        unsigned long long hostCount[8] = {0};
        for (int c = 0; c < 8; ++c)
            for (int b = 0; b < kBandSlots; ++b) hostCount[c] += bandCount[c * kBandSlots + b];
        // class segments are padded to whole tiles of kPairTile events
        int64_t base[8] = {0}, sortedStart[8] = {0};
        int64_t total = 0, seen = 0;
        for (int c = 0; c < kFakeClasses; ++c) {
            base[c] = total;
            sortedStart[c] = seen;
            seen += (int64_t)hostCount[c];
            int64_t inClass = 0;
            for (int b = 0; b < kMassBands; ++b) {
                e->fakeBandStart[c][b] = inClass;
                inClass += (int64_t)bandCount[c * kBandSlots + b];
            }
            e->fakeClassBase[c] = total;
            e->fakeClassReal[c] = (int64_t)hostCount[c];
            e->fakeClassCount[c] = ((int64_t)hostCount[c] + kPairTile - 1) / kPairTile * kPairTile;
            total += e->fakeClassCount[c];
        }
        sortedStart[kIrregularClass] = seen;
        e->fakeIrregularCount = (int64_t)hostCount[kIrregularClass];
        e->fakeEvents.reserve(total > 0 ? total : 1);
        e->fakeFilterTiles.reserve(total > 0 ? total / kPairTile : 1);
        e->fakeIrregular.reserve(e->fakeIrregularCount > 0 ? e->fakeIrregularCount : 1);
        if (count > 0) {
            CUDA_CHECK(cudaMemcpyAsync(baseDev, base, sizeof(base), cudaMemcpyHostToDevice, e->stream));
            CUDA_CHECK(cudaMemcpyAsync(startDev, sortedStart, sizeof(sortedStart), cudaMemcpyHostToDevice, e->stream));
            kFakeGather<<<ceilDiv(count, 256), 256, 0, e->stream>>>(raw, count, keysOut, indexOut, startDev, baseDev,
                                                                  e->fakeEvents.get(), e->fakeFilterTiles.get(),
                                                                  e->fakeIrregular.get());
            e->launched();
        }
        for (int c = 0; c < kFakeClasses; ++c) {
            const int64_t pad = e->fakeClassCount[c] - e->fakeClassReal[c];
            if (pad > 0) {
                kFakePadEvents<<<ceilDiv(pad, 128), 128, 0, e->stream>>>(e->fakeEvents.get(), e->fakeFilterTiles.get(),
                                                                       e->fakeClassBase[c], e->fakeClassReal[c],
                                                                       e->fakeClassCount[c]);
                e->launched();
            }
        }
        CUDA_CHECK(cudaStreamSynchronize(e->stream));          // the arena goes out of scope; host arrays were read
        e->fakeEventCount = count;
        e->hmc.gradCacheReady = false;                         // the gradients kept belong to the old sample
    });
}

int smcmc_unbinned_set_events(smcmc_engine* e, const smcmc_event* events, int64_t count) {
    return guarded(e, [&]() {
        if (e->cfg.likelihood != SMCMC_LLH_UNBINNED) throw Error(SMCMC_ERR_LOGIC, "engine was not created with SMCMC_LLH_UNBINNED");
        if (count < 0 || (count > 0 && !events)) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "bad event array");
        if (count > 0xffffffffLL) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "more than 2^32 events per engine");
        e->unbEvents.reserve(count > 0 ? count : 1);
        unsigned long long tagged = 0;
        if (count > 0) {
            size_t sortBytes = 0;
            CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, sortBytes, (unsigned long long*)nullptr,
                                                       (unsigned long long*)nullptr, (unsigned int*)nullptr,
                                                       (unsigned int*)nullptr, (int)count, 0, 33, e->stream));
            auto align = [](size_t b) { return (b + 255) / 256 * 256; };
            const size_t n = (size_t)count;
            const size_t offKeysIn = align(n * sizeof(smcmc_event)), offKeysOut = offKeysIn + align(n * 8);
            const size_t offIndexIn = offKeysOut + align(n * 8), offIndexOut = offIndexIn + align(n * 4);
            const size_t offSort = offIndexOut + align(n * 4), offSmall = offSort + align(sortBytes);
            DeviceBuffer<unsigned char> arena;
            arena.reserve(offSmall + 256);
            unsigned char* b0 = arena.get();
            smcmc_event* raw = (smcmc_event*)b0;
            unsigned long long* keysIn = (unsigned long long*)(b0 + offKeysIn);
            unsigned long long* keysOut = (unsigned long long*)(b0 + offKeysOut);
            unsigned int* indexIn = (unsigned int*)(b0 + offIndexIn);
            unsigned int* indexOut = (unsigned int*)(b0 + offIndexOut);
            unsigned long long* counter = (unsigned long long*)(b0 + offSmall);
            CUDA_CHECK(cudaMemsetAsync(counter, 0, 8, e->stream));
            CUDA_CHECK(cudaMemcpyAsync(raw, events, sizeof(smcmc_event) * count, cudaMemcpyHostToDevice, e->stream));
            kUnbinnedSortKeys<<<ceilDiv(count, 256), 256, 0, e->stream>>>(raw, count, keysIn, indexIn, counter);
            e->launched();
            CUDA_CHECK(cub::DeviceRadixSort::SortPairs(b0 + offSort, sortBytes, keysIn, keysOut, indexIn, indexOut,
                                                       (int)count, 0, 33, e->stream));
            e->launched();
            kUnbinnedGather<<<ceilDiv(count, 256), 256, 0, e->stream>>>(raw, count, indexOut, e->unbEvents.get());
            e->launched();
            CUDA_CHECK(cudaMemcpyAsync(&tagged, counter, 8, cudaMemcpyDeviceToHost, e->stream));
            CUDA_CHECK(cudaStreamSynchronize(e->stream));
        }
        e->unbClassCount[0] = count - (int64_t)tagged;
        e->unbClassCount[1] = (int64_t)tagged;
        e->unbEventCount = count;
        e->hmc.gradCacheReady = false;                 // the gradients kept belong to the old sample
    });
}

int smcmc_fake_set_data(smcmc_engine* e, const double* data150, double exposure) {
    return guarded(e, [&]() {
        if (e->cfg.likelihood != SMCMC_LLH_FAKE && e->cfg.likelihood != SMCMC_LLH_FAKE2)
            throw Error(SMCMC_ERR_LOGIC, "engine was not created with SMCMC_LLH_FAKE or SMCMC_LLH_FAKE2");
        if (!data150) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null data histograms");
        CUDA_CHECK(cudaMemcpyAsync(e->fakeData.get(), data150, 150 * sizeof(double), cudaMemcpyHostToDevice, e->stream));
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        e->fakeExposure = exposure;
        e->fakeDataSet = true;
        e->hmc.gradCacheReady = false;                 // the gradients kept belong to the old data
    });
}

int smcmc_dummy_set_mode(smcmc_engine* e, int mode) {
    return guarded(e, [&]() {
        if (e->cfg.likelihood != SMCMC_LLH_DUMMY) throw Error(SMCMC_ERR_LOGIC, "engine was not created with SMCMC_LLH_DUMMY");
        if (mode != SMCMC_DUMMY_EXACT && mode != SMCMC_DUMMY_TENSOR) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "unknown mode");
        e->dummyMode = mode;
        e->hmc.gradCacheReady = false;                 // (kHmcLeapCached: gradients kept from the other mode's arithmetic)
    });
}

int smcmc_dummy_set_error(smcmc_engine* e, const double* err, int nn) {
    return guarded(e, [&]() {
        if (e->cfg.likelihood != SMCMC_LLH_DUMMY) throw Error(SMCMC_ERR_LOGIC, "engine was not created with SMCMC_LLH_DUMMY");
        if (!err || nn != e->n()) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "error matrix must be dim x dim");
        e->errMatrix.reserve((size_t)nn * nn);
        e->errMatrixT.reserve((size_t)nn * nn);
        std::vector<double> t((size_t)nn * nn);
        for (int i = 0; i < nn; ++i)
            for (int j = 0; j < nn; ++j) t[(size_t)i * nn + j] = err[(size_t)j * nn + i];
        CUDA_CHECK(cudaMemcpyAsync(e->errMatrix.get(), err, sizeof(double) * nn * nn, cudaMemcpyHostToDevice, e->stream));
        CUDA_CHECK(cudaMemcpyAsync(e->errMatrixT.get(), t.data(), sizeof(double) * nn * nn, cudaMemcpyHostToDevice, e->stream));
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        e->hmc.gradCacheReady = false;                 // the gradients kept belong to the old matrix
        e->errDim = nn;
    });
}

static void evalHost(smcmc_engine* e, const double* x, int m, double* llh, double* hist) {
    if (m < 1 || !x) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "bad point array");
    const size_t n = e->n();
    e->evalX.reserve((size_t)m * n);
    e->evalOut.reserve(m);
    if (hist) e->evalHist.reserve((size_t)m * 150);
    CUDA_CHECK(cudaMemcpyAsync(e->evalX.get(), x, sizeof(double) * m * n, cudaMemcpyHostToDevice, e->stream));
    e->evaluate(e->evalX.get(), m, e->evalOut.get(), hist ? e->evalHist.get() : nullptr);
    if (llh) CUDA_CHECK(cudaMemcpyAsync(llh, e->evalOut.get(), sizeof(double) * m, cudaMemcpyDeviceToHost, e->stream));
    if (hist) CUDA_CHECK(cudaMemcpyAsync(hist, e->evalHist.get(), sizeof(double) * m * 150, cudaMemcpyDeviceToHost, e->stream));
    CUDA_CHECK(cudaStreamSynchronize(e->stream));
}

int smcmc_fake_histograms(smcmc_engine* e, const double* x, int m, double* out) {
    return guarded(e, [&]() {
        if (e->cfg.likelihood != SMCMC_LLH_FAKE && e->cfg.likelihood != SMCMC_LLH_FAKE2)
            throw Error(SMCMC_ERR_LOGIC, "engine was not created with SMCMC_LLH_FAKE or SMCMC_LLH_FAKE2");
        if (!out) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null output");
        evalHost(e, x, m, nullptr, out);
    });
}

int smcmc_fake_counts(smcmc_engine* e, const double* x, int m, uint32_t* out) {
    return guarded(e, [&]() {
        if (e->cfg.likelihood != SMCMC_LLH_FAKE && e->cfg.likelihood != SMCMC_LLH_FAKE2)
            throw Error(SMCMC_ERR_LOGIC, "engine was not created with SMCMC_LLH_FAKE or SMCMC_LLH_FAKE2");
        if (!out) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null output");
        e->wantFullCounts = true;
        try { evalHost(e, x, m, nullptr, nullptr); } catch (...) { e->wantFullCounts = false; throw; }
        e->wantFullCounts = false;
        const int stride = e->fakeCountStride;
        std::vector<uint32_t> host((size_t)kFakeSlots * stride);
        CUDA_CHECK(cudaMemcpyAsync(host.data(), e->fakeCounts.get(), host.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->stream));
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        for (int p = 0; p < m; ++p)
            for (int s = 0; s < kFakeSlots; ++s) out[(size_t)p * kFakeSlots + s] = host[(size_t)s * stride + p];
    });
}

int smcmc_fake_filter_check(smcmc_engine* e, const double* x, int m, uint64_t* out3) {
    return guarded(e, [&]() {
        if (e->cfg.likelihood != SMCMC_LLH_FAKE && e->cfg.likelihood != SMCMC_LLH_FAKE2)
            throw Error(SMCMC_ERR_LOGIC, "engine was not created with SMCMC_LLH_FAKE or SMCMC_LLH_FAKE2");
        if (!out3) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null output");
        e->wantFullCounts = true;
        try { evalHost(e, x, m, nullptr, nullptr); } catch (...) { e->wantFullCounts = false; throw; }   // fills the per-chain constants for these points
        e->wantFullCounts = false;
        PairLaunch L = e->pairLaunch(m, e->fakeCountStride);
        CUDA_CHECK(cudaMemsetAsync(e->fakeStats.get(), 0, 4 * sizeof(unsigned long long), e->stream));
        dim3 grid(512, ceilDiv(m, 128));
        kFakeVerifyFilter<<<grid, 128, 0, e->stream>>>(L, e->fakeStats.get());
        e->launched();
        unsigned long long host[4];
        CUDA_CHECK(cudaMemcpyAsync(host, e->fakeStats.get(), sizeof(host), cudaMemcpyDeviceToHost, e->stream));
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        for (int i = 0; i < 3; ++i) out3[i] = host[i];
    });
}

int smcmc_fake_skip_check(smcmc_engine* e, const double* x, int m, uint64_t* out3) {
    return guarded(e, [&]() {
        if (e->cfg.likelihood != SMCMC_LLH_FAKE && e->cfg.likelihood != SMCMC_LLH_FAKE2)
            throw Error(SMCMC_ERR_LOGIC, "engine was not created with SMCMC_LLH_FAKE or SMCMC_LLH_FAKE2");
        if (!out3) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null output");
        e->wantFullCounts = true;
        try { evalHost(e, x, m, nullptr, nullptr); } catch (...) { e->wantFullCounts = false; throw; }   // fills the per-chain constants for these points
        e->wantFullCounts = false;
        PairLaunch L = e->pairLaunch(m, e->fakeCountStride);
        CUDA_CHECK(cudaMemsetAsync(e->fakeStats.get(), 0, 4 * sizeof(unsigned long long), e->stream));
        dim3 grid(256, ceilDiv(m, 128));
        kFakeSkipCheck<<<grid, 128, 0, e->stream>>>(L, e->fakeStats.get());
        e->launched();
        unsigned long long host[4];
        CUDA_CHECK(cudaMemcpyAsync(host, e->fakeStats.get(), sizeof(host), cudaMemcpyDeviceToHost, e->stream));
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        for (int i = 0; i < 3; ++i) out3[i] = host[i];
    });
}

int smcmc_eval(smcmc_engine* e, const double* x, int m, double* llh) {
    return guarded(e, [&]() {
        if (!llh) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null output");
        evalHost(e, x, m, llh, nullptr);
    });
}

int smcmc_start(smcmc_engine* e, const double* x0, int32_t* ok) {
    return guarded(e, [&]() {
        if (!x0) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null starting points");
        const size_t bytes = sizeof(double) * e->E() * e->n();
        e->vaatSynced = false;
        CUDA_CHECK(cudaMemcpyAsync(e->xAcc.get(), x0, bytes, cudaMemcpyHostToDevice, e->stream));   // :247-256
        CUDA_CHECK(cudaMemcpyAsync(e->xProp.get(), e->xAcc.get(), bytes, cudaMemcpyDeviceToDevice, e->stream));
        e->evaluate(e->xProp.get(), e->E(), e->llhProp.get(), nullptr);                             // :258
        if (e->propKind == SMCMC_PROPOSAL_VAAT) {
            if (e->pooledEvery > 0) throw Error(SMCMC_ERR_LOGIC, "pooled adaptation belongs to the adaptive proposal");
            PropSettings psv = e->settings();
            if (!e->started) e->vaatAllocate();
            if (!e->vaatInitialized) e->vaatWindow = 100;                                           // InitializeState (first Start only), TProposeVAATStep.H:197-208
            e->vaatInitialized = true;
            kStoreStartLlh<<<ceilDiv(e->E(), 128), 128, 0, e->stream>>>(e->sc.get(), e->llhProp.get(), e->E());
            e->launched();
            kVaatInit<<<ceilDiv(e->E(), 128), 128, 0, e->stream>>>(e->arrays(), e->vaatArrays(), e->E(), e->n(), e->okDev.get());
            e->launched();
            (void)psv;
            std::vector<int32_t> okv(e->E());
            CUDA_CHECK(cudaMemcpyAsync(okv.data(), e->okDev.get(), sizeof(int32_t) * e->E(), cudaMemcpyDeviceToHost, e->stream));
            CUDA_CHECK(cudaStreamSynchronize(e->stream));
            if (ok) std::memcpy(ok, okv.data(), sizeof(int32_t) * e->E());
            e->started = true;
            return;
        }
        e->resolveInitDefaults();
        e->resolveResetDefaults();
        PropSettings ps = e->settings();
        // stash the start likelihood in the chain records
        kStoreStartLlh<<<ceilDiv(e->E(), 128), 128, 0, e->stream>>>(e->sc.get(), e->llhProp.get(), e->E());
        e->launched();
        kInitState<<<ceilDiv(e->E(), kWarpsPerBlock), kWarpsPerBlock * 32, 0, e->stream>>>(e->arrays(), ps, e->E(), e->okDev.get());
        e->launched();
        std::vector<int32_t> okHost(e->E());
        CUDA_CHECK(cudaMemcpyAsync(okHost.data(), e->okDev.get(), sizeof(int32_t) * e->E(), cudaMemcpyDeviceToHost, e->stream));
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        if (ok) std::memcpy(ok, okHost.data(), sizeof(int32_t) * e->E());
        e->started = true;
        e->checkChainStatus();
        if (e->pooledEvery > 0 && e->poolStats.count() == 0) e->poolInit();
    });
}

int smcmc_step(smcmc_engine* e, int nsteps, int metropolis) {
    return guarded(e, [&]() {
        requireStarted(e);
        e->stepMany(nsteps, metropolis);
    });
}

int smcmc_step_trace(smcmc_engine* e, int nsteps, int metropolis, const smcmc_trace* trace) {
    return guarded(e, [&]() {
        requireStarted(e);
        if (nsteps < 1) return;
        const size_t rows = (size_t)nsteps * e->E();
        DeviceBuffer<int32_t> acc;
        DeviceBuffer<double> la, lp, pts, sg, rms;
        TraceDev tr = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
        if (trace) {
            if (trace->accepted) { acc.reserve(rows); tr.accepted = acc.get(); }
            if (trace->llh_accepted) { la.reserve(rows); tr.llhAccepted = la.get(); }
            if (trace->llh_proposed) { lp.reserve(rows); tr.llhProposed = lp.get(); }
            if (trace->points) { pts.reserve(rows * e->n()); tr.points = pts.get(); }
            if (trace->sigma) { sg.reserve(rows); tr.sigma = sg.get(); }
            if (trace->step_rms) { rms.reserve(rows); tr.stepRMS = rms.get(); }
        }
        for (int s = 0; s < nsteps; ++s) e->stepOnce(metropolis, tr, s);
        if (trace) {
            if (trace->accepted) CUDA_CHECK(cudaMemcpyAsync(trace->accepted, acc.get(), rows * sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
            if (trace->llh_accepted) CUDA_CHECK(cudaMemcpyAsync(trace->llh_accepted, la.get(), rows * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
            if (trace->llh_proposed) CUDA_CHECK(cudaMemcpyAsync(trace->llh_proposed, lp.get(), rows * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
            if (trace->points) CUDA_CHECK(cudaMemcpyAsync(trace->points, pts.get(), rows * e->n() * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
            if (trace->sigma) CUDA_CHECK(cudaMemcpyAsync(trace->sigma, sg.get(), rows * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
            if (trace->step_rms) CUDA_CHECK(cudaMemcpyAsync(trace->step_rms, rms.get(), rows * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
        }
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        e->checkChainStatus();
    });
}

int smcmc_save_state(smcmc_engine* e, const smcmc_saved_state* out) {
    return guarded(e, [&]() {
        requireStarted(e);
        if (e->propKind == SMCMC_PROPOSAL_VAAT)
            throw Error(SMCMC_ERR_LOGIC, "TProposeVAATStep does not save or restore its state (TProposeVAATStep.H:33-36)");
        if (!out) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null state");
        const size_t E = e->E(), n = e->n(), tri = e->tri();
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        std::vector<ChainScalars> h(E);
        CUDA_CHECK(cudaMemcpy(h.data(), e->sc.get(), sizeof(ChainScalars) * E, cudaMemcpyDeviceToHost));
        if (out->accepted) CUDA_CHECK(cudaMemcpy(out->accepted, e->xAcc.get(), E * n * 8, cudaMemcpyDeviceToHost));
        if (out->central_point) CUDA_CHECK(cudaMemcpy(out->central_point, e->center.get(), E * n * 8, cudaMemcpyDeviceToHost));
        if (out->covariance)
            CUDA_CHECK(cudaMemcpy2D(out->covariance, tri * 8, e->cov.get(), (size_t)e->covStride * 8, tri * 8, E,
                                    cudaMemcpyDeviceToHost));
        if (out->covariance_trace) {
            DeviceBuffer<double> tr;
            tr.reserve(E);
            kCovarianceTrace<<<ceilDiv((long long)E, 128), 128, 0, e->stream>>>(e->cov.get(), e->covStride, (int)E, (int)n, tr.get());
            e->launched();
            CUDA_CHECK(cudaMemcpyAsync(out->covariance_trace, tr.get(), E * 8, cudaMemcpyDeviceToHost, e->stream));
            CUDA_CHECK(cudaStreamSynchronize(e->stream));
        }
        for (size_t c = 0; c < E; ++c) {
            if (out->log_likelihood) out->log_likelihood[c] = h[c].accLlh;
            if (out->total_steps) out->total_steps[c] = h[c].totalSteps;
            if (out->step_rms) out->step_rms[c] = h[c].stepRMS;
            if (out->trials) out->trials[c] = h[c].trials;
            if (out->successes) out->successes[c] = h[c].successes;
            if (out->next_update) out->next_update[c] = h[c].nextUpdate;
            if (out->acceptance) out->acceptance[c] = h[c].acceptance;
            if (out->acceptance_trials) out->acceptance_trials[c] = h[c].acceptanceTrials;
            if (out->sigma) out->sigma[c] = h[c].sigma;
            if (out->central_point_trials) out->central_point_trials[c] = h[c].centerTrials;
            if (out->covariance_trials) out->covariance_trials[c] = h[c].covTrials;
        }
    });
}

int smcmc_restore_state(smcmc_engine* e, const smcmc_saved_state* in, int32_t* mismatch) {
    return guarded(e, [&]() {
        requireStarted(e);
        if (e->propKind == SMCMC_PROPOSAL_VAAT)
            throw Error(SMCMC_ERR_LOGIC, "TProposeVAATStep does not save or restore its state (TProposeVAATStep.H:33-36)");
        if (!in || !in->accepted || !in->log_likelihood || !in->total_steps || !in->step_rms || !in->trials ||
            !in->successes || !in->next_update || !in->acceptance || !in->acceptance_trials || !in->sigma ||
            !in->central_point || !in->central_point_trials || !in->covariance || !in->covariance_trials)
            throw Error(SMCMC_ERR_LOGIC, "Past the end of the covariance");      // incomplete saved state (:1572-1576)
        if (e->pooledEvery > 0) throw Error(SMCMC_ERR_LOGIC, "restore is defined for per-chain adaptation");
        const size_t E = e->E(), n = e->n(), tri = e->tri();
        DeviceBuffer<double> d[7];
        DeviceBuffer<int> i4[4];
        DeviceBuffer<int32_t> mm;
        auto upD = [&](DeviceBuffer<double>& b, const double* src) {
            b.reserve(E);
            CUDA_CHECK(cudaMemcpyAsync(b.get(), src, E * 8, cudaMemcpyHostToDevice, e->stream));
            return b.get();
        };
        auto upI = [&](DeviceBuffer<int>& b, const int32_t* src) {
            b.reserve(E);
            CUDA_CHECK(cudaMemcpyAsync(b.get(), src, E * 4, cudaMemcpyHostToDevice, e->stream));
            return b.get();
        };
        e->vaatSynced = false;
        CUDA_CHECK(cudaMemcpyAsync(e->xAcc.get(), in->accepted, E * n * 8, cudaMemcpyHostToDevice, e->stream));
        CUDA_CHECK(cudaMemcpyAsync(e->center.get(), in->central_point, E * n * 8, cudaMemcpyHostToDevice, e->stream));
        CUDA_CHECK(cudaMemcpy2DAsync(e->cov.get(), (size_t)e->covStride * 8, in->covariance, tri * 8, tri * 8, E,
                                     cudaMemcpyHostToDevice, e->stream));
        RestoreScalars r;
        r.savedLlh = upD(d[0], in->log_likelihood);
        r.stepRMS = upD(d[1], in->step_rms);
        r.acceptance = upD(d[2], in->acceptance);
        r.acceptanceTrials = upD(d[3], in->acceptance_trials);
        r.sigma = upD(d[4], in->sigma);
        r.centerTrials = upD(d[5], in->central_point_trials);
        r.covTrials = upD(d[6], in->covariance_trials);
        r.totalSteps = upI(i4[0], in->total_steps);
        r.trials = upI(i4[1], in->trials);
        r.successes = upI(i4[2], in->successes);
        r.nextUpdate = upI(i4[3], in->next_update);
        e->evaluate(e->xAcc.get(), e->E(), e->llhProp.get(), nullptr);                    // :335
        mm.reserve(E);
        PropSettings ps = e->settings();
        kRestore<<<ceilDiv(e->E(), kWarpsPerBlock), kWarpsPerBlock * 32, 0, e->stream>>>(e->arrays(), ps, e->E(), r,
                                                                                         e->llhProp.get(), mm.get());
        e->launched();
        if (mismatch) CUDA_CHECK(cudaMemcpyAsync(mismatch, mm.get(), E * 4, cudaMemcpyDeviceToHost, e->stream));
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        e->checkChainStatus();
    });
}

int smcmc_get_step_index(smcmc_engine* e, uint32_t* step) {
    return guarded(e, [&]() {
        if (!step) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null output");
        *step = e->stepIndex;
    });
}

int smcmc_set_step_index(smcmc_engine* e, uint32_t step) {
    return guarded(e, [&]() { e->stepIndex = step; });
}

int smcmc_get(smcmc_engine* e, int field, void* dst, size_t bytes) {
    return guarded(e, [&]() {
        if (!dst) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null destination");
        const size_t E = e->E(), n = e->n();
        auto need = [&](size_t want) {
            if (bytes < want) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "destination too small");
        };
        auto copyArray = [&](const void* src, size_t want) {
            need(want);
            CUDA_CHECK(cudaMemcpyAsync(dst, src, want, cudaMemcpyDeviceToHost, e->stream));
            CUDA_CHECK(cudaStreamSynchronize(e->stream));
        };
        const bool vaat = e->propKind == SMCMC_PROPOSAL_VAAT;
        if (field >= SMCMC_F_VAAT_SIGMA && field <= SMCMC_F_VAAT_QUEUE && (!vaat || !e->started))
            throw Error(SMCMC_ERR_LOGIC, "the sampler was not started with SMCMC_PROPOSAL_VAAT");
        if (vaat && e->started && (field == SMCMC_F_ACCEPTANCE || field == SMCMC_F_VAAT_LAST_INDEX || field == SMCMC_F_VAAT_QUEUE)) {
            if (field == SMCMC_F_ACCEPTANCE) {                                // GetAcceptance, TProposeVAATStep.H:155-163
                need(E * 8);
                std::vector<double> acc(E * n);
                CUDA_CHECK(cudaMemcpyAsync(acc.data(), e->vAcceptance.get(), acc.size() * 8, cudaMemcpyDeviceToHost, e->stream));
                CUDA_CHECK(cudaStreamSynchronize(e->stream));
                for (size_t c = 0; c < E; ++c) {
                    double t = 0.0;
                    for (size_t i = 0; i < n; ++i) t += acc[c * n + i];
                    ((double*)dst)[c] = t / (double)n;
                }
                return;
            }
            need(E * 4);
            std::vector<VaatState> st(E);
            CUDA_CHECK(cudaMemcpyAsync(st.data(), e->vState.get(), E * sizeof(VaatState), cudaMemcpyDeviceToHost, e->stream));
            CUDA_CHECK(cudaStreamSynchronize(e->stream));
            for (size_t c = 0; c < E; ++c)
                ((int32_t*)dst)[c] = field == SMCMC_F_VAAT_LAST_INDEX ? st[c].lastIndex : st[c].queueSize;
            return;
        }
        switch (field) {
        case SMCMC_F_VAAT_SIGMA: copyArray(e->vSigma.get(), E * n * 8); return;
        case SMCMC_F_VAAT_ACCEPTANCE: copyArray(e->vAcceptance.get(), E * n * 8); return;
        case SMCMC_F_VAAT_ACCEPTANCE_TRIALS: copyArray(e->vAccTrials.get(), E * n * 4); return;
        case SMCMC_F_ACCEPTANCE_WINDOW:
            if (vaat) { need(8); *(double*)dst = e->vaatWindow; return; }
            break;
        default: break;
        }
        switch (field) {
        case SMCMC_F_ACCEPTED: copyArray(e->xAcc.get(), E * n * 8); return;
        case SMCMC_F_PROPOSED: copyArray(e->xProp.get(), E * n * 8); return;
        case SMCMC_F_CENTER: copyArray(e->center.get(), E * n * 8); return;
        case SMCMC_F_COVARIANCE:
            need(E * e->tri() * 8);
            CUDA_CHECK(cudaMemcpy2DAsync(dst, (size_t)e->tri() * 8, e->cov.get(), (size_t)e->covStride * 8,
                                         (size_t)e->tri() * 8, E, cudaMemcpyDeviceToHost, e->stream));
            CUDA_CHECK(cudaStreamSynchronize(e->stream));
            return;
        case SMCMC_F_DECOMPOSITION: copyArray(e->decomp.get(), E * n * n * 8); return;
        case SMCMC_F_COVARIANCE_WINDOW: need(8); *(double*)dst = e->covWindow; return;
        case SMCMC_F_ACCEPTANCE_WINDOW: need(8); *(double*)dst = e->accWindow; return;
        case SMCMC_F_TARGET_ACCEPTANCE: need(8); *(double*)dst = e->target; return;
        case SMCMC_F_POOLED_MEAN:
            if (!e->poolMean.count()) throw Error(SMCMC_ERR_LOGIC, "pooled adaptation is off");
            copyArray(e->poolMean.get(), n * 8); return;
        case SMCMC_F_POOLED_COVARIANCE:
            if (!e->poolCov.count()) throw Error(SMCMC_ERR_LOGIC, "pooled adaptation is off");
            copyArray(e->poolCov.get(), e->tri() * 8); return;
        case SMCMC_F_POOLED_DECOMPOSITION:
            if (!e->poolDecomp.count()) throw Error(SMCMC_ERR_LOGIC, "pooled adaptation is off");
            copyArray(e->poolDecomp.get(), n * n * 8); return;
        case SMCMC_F_POOLED_COUNT:
            if (!e->poolStatsAll.count()) throw Error(SMCMC_ERR_LOGIC, "pooled adaptation is off");
            copyArray(e->poolStatsAll.get(), 8); return;
        default: break;
        }
        std::vector<ChainScalars> h(E);
        CUDA_CHECK(cudaMemcpyAsync(h.data(), e->sc.get(), sizeof(ChainScalars) * E, cudaMemcpyDeviceToHost, e->stream));
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        auto putD = [&](double ChainScalars::*m) {
            need(E * 8);
            for (size_t c = 0; c < E; ++c) ((double*)dst)[c] = h[c].*m;
        };
        auto putI = [&](int ChainScalars::*m) {
            need(E * 4);
            for (size_t c = 0; c < E; ++c) ((int32_t*)dst)[c] = h[c].*m;
        };
        switch (field) {
        case SMCMC_F_ACCEPTED_LLH: putD(&ChainScalars::accLlh); break;
        case SMCMC_F_PROPOSED_LLH: putD(&ChainScalars::propLlh); break;
        case SMCMC_F_STEP_RMS: putD(&ChainScalars::stepRMS); break;
        case SMCMC_F_SIGMA: putD(&ChainScalars::sigma); break;
        case SMCMC_F_SIGMA_TRACE: putD(&ChainScalars::sigmaTrace); break;
        case SMCMC_F_ACCEPTANCE: putD(&ChainScalars::acceptance); break;
        case SMCMC_F_ACCEPTANCE_TRIALS: putD(&ChainScalars::acceptanceTrials); break;
        case SMCMC_F_ACCEPTANCE_RIGIDITY: putD(&ChainScalars::rigidity); break;
        case SMCMC_F_COVARIANCE_TRIALS: putD(&ChainScalars::covTrials); break;
        case SMCMC_F_CENTER_TRIALS: putD(&ChainScalars::centerTrials); break;
        case SMCMC_F_TRIALS: putI(&ChainScalars::trials); break;
        case SMCMC_F_SUCCESSES: putI(&ChainScalars::successes); break;
        case SMCMC_F_NEXT_UPDATE: putI(&ChainScalars::nextUpdate); break;
        case SMCMC_F_TOTAL_STEPS: putI(&ChainScalars::totalSteps); break;
        case SMCMC_F_LLH_CALLS: putI(&ChainScalars::llhCalls); break;
        case SMCMC_F_STATUS: putI(&ChainScalars::status); break;
        case SMCMC_F_COVARIANCE_TRACE: {                                    // :961-967
            need(E * 8);
            DeviceBuffer<double> tr;
            tr.reserve(E);
            kCovarianceTrace<<<ceilDiv((long long)E, 128), 128, 0, e->stream>>>(e->cov.get(), e->covStride, (int)E, (int)n, tr.get());
            e->launched();
            CUDA_CHECK(cudaMemcpyAsync(dst, tr.get(), E * 8, cudaMemcpyDeviceToHost, e->stream));
            CUDA_CHECK(cudaStreamSynchronize(e->stream));
            break;
        }
        default: throw Error(SMCMC_ERR_INVALID_ARGUMENT, "unknown field");
        }
    });
}

namespace smcmc {
// 8 independent DFMA chains per thread, 4096 iterations.
__global__ void __launch_bounds__(256) kFp64Peak(double* out, double a, double b, int iters) {
    double v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = (double)(threadIdx.x + k);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = __fma_rn(v[k], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += v[k];
    if (s == 12345.678) out[0] = s;      // never true: keeps the chain alive
}
}  // namespace smcmc

int smcmc_measure_fp64_peak(int device, double* tflops) {
    return guarded(nullptr, [&]() {
        if (!tflops) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null output");
        int count = 0;
        if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
            cudaGetLastError();
            throw Error(SMCMC_ERR_NO_DEVICE, "no CUDA device");
        }
        CUDA_CHECK(cudaSetDevice(device));
        cudaDeviceProp prop;
        CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
        DeviceBuffer<double> out;
        out.reserve(1);
        const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
        cudaEvent_t e0, e1;
        CUDA_CHECK(cudaEventCreate(&e0));
        CUDA_CHECK(cudaEventCreate(&e1));
        double best = 0.0;
        for (int rep = 0; rep < 6; ++rep) {
            CUDA_CHECK(cudaEventRecord(e0));
            kFp64Peak<<<blocks, threads>>>(out.get(), 0.999999, 1e-7, iters);
            CUDA_CHECK(cudaEventRecord(e1));
            CUDA_CHECK(cudaEventSynchronize(e1));
            float ms = 0.f;
            CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
            double flops = 2.0 * 8.0 * iters * (double)blocks * threads;
            if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
        }
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        *tflops = best;
    });
}

namespace smcmc {
// 8 independent DMMA (mma.sync.m8n8k4.f64) accumulator chains per warp, operands in registers.
__global__ void __launch_bounds__(256) kDmmaPeak(double* out, double a, double b, int iters) {
    double acc[8][2];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k][0] = acc[k][1] = (double)(threadIdx.x + k);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) dmma884(acc[k][0], acc[k][1], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += acc[k][0] + acc[k][1];
    if (s == 12345.678) out[0] = s;      // never true: keeps the chains alive
}
}  // namespace smcmc

int smcmc_measure_dmma_peak(int device, double* tflops) {
    return guarded(nullptr, [&]() {
        if (!tflops) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null output");
        int count = 0;
        if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
            cudaGetLastError();
            throw Error(SMCMC_ERR_NO_DEVICE, "no CUDA device");
        }
        CUDA_CHECK(cudaSetDevice(device));
        cudaDeviceProp prop;
        CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
        DeviceBuffer<double> out;
        out.reserve(1);
        const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 2048;
        cudaEvent_t e0, e1;
        CUDA_CHECK(cudaEventCreate(&e0));
        CUDA_CHECK(cudaEventCreate(&e1));
        double best = 0.0;
        for (int rep = 0; rep < 6; ++rep) {
            CUDA_CHECK(cudaEventRecord(e0));
            kDmmaPeak<<<blocks, threads>>>(out.get(), 0.999999, 1e-7, iters);
            CUDA_CHECK(cudaEventRecord(e1));
            CUDA_CHECK(cudaEventSynchronize(e1));
            float ms = 0.f;
            CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
            // one m8n8k4 DMMA per warp = 8 x 8 x 4 multiply-adds = 512 flop
            const double flops = 512.0 * 8.0 * iters * (double)blocks * (threads / 32);
            if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
        }
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        *tflops = best;
    });
}

namespace smcmc {
// 8 independent MUFU.EX2 chains per thread.
__global__ void __launch_bounds__(256) kSfuPeak(float* out, float a, int iters) {
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = a * (float)(threadIdx.x + k);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(v[k]));
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += v[k];
    if (s == 12345.678f) out[0] = s;     // never true: keeps the chains alive
}
}  // namespace smcmc

int smcmc_selftest_division(int device, int64_t count, uint64_t seed, int64_t* mismatches) {
    return guarded(nullptr, [&]() {
        if (!mismatches || count < 0) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "bad arguments");
        int devices = 0;
        if (cudaGetDeviceCount(&devices) != cudaSuccess || device < 0 || device >= devices) {
            cudaGetLastError();
            throw Error(SMCMC_ERR_NO_DEVICE, "no CUDA device");
        }
        CUDA_CHECK(cudaSetDevice(device));
        DeviceBuffer<unsigned long long> bad;
        bad.reserve(1);
        CUDA_CHECK(cudaMemset(bad.get(), 0, sizeof(unsigned long long)));
        kSelftestDivision<<<148 * 8, 256>>>(seed, (long long)count, bad.get());
        CUDA_CHECK(cudaGetLastError());
        unsigned long long h = 0;
        CUDA_CHECK(cudaMemcpy(&h, bad.get(), sizeof h, cudaMemcpyDeviceToHost));
        *mismatches = (int64_t)h;
    });
}

int smcmc_measure_sfu_peak(int device, double* gops) {
    return guarded(nullptr, [&]() {
        if (!gops) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null output");
        int count = 0;
        if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
            cudaGetLastError();
            throw Error(SMCMC_ERR_NO_DEVICE, "no CUDA device");
        }
        CUDA_CHECK(cudaSetDevice(device));
        cudaDeviceProp prop;
        CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
        DeviceBuffer<float> out;
        out.reserve(1);
        const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 2048;
        cudaEvent_t e0, e1;
        CUDA_CHECK(cudaEventCreate(&e0));
        CUDA_CHECK(cudaEventCreate(&e1));
        double best = 0.0;
        for (int rep = 0; rep < 6; ++rep) {
            CUDA_CHECK(cudaEventRecord(e0));
            kSfuPeak<<<blocks, threads>>>(out.get(), 1e-3f, iters);
            CUDA_CHECK(cudaEventRecord(e1));
            CUDA_CHECK(cudaEventSynchronize(e1));
            float ms = 0.f;
            CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
            const double ops = 8.0 * iters * (double)blocks * threads;
            if (rep > 0) best = std::max(best, ops / (ms * 1e-3) / 1e9);
        }
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        *gops = best;
    });
}

int64_t smcmc_launch_count(const smcmc_engine* e) { return e ? e->launches : 0; }

int smcmc_enable_kernel_timing(smcmc_engine* e, int on) {
    return guarded(e, [&]() { e->timing = on != 0; });
}

int smcmc_diag_enable(smcmc_engine* e, int max_lag) {
    return guarded(e, [&]() {
        if (max_lag < 0) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "max_lag must not be negative");
        const size_t En = (size_t)e->E() * e->n();
        if ((size_t)max_lag * En * sizeof(double) > ((size_t)48 << 30))
            throw Error(SMCMC_ERR_INVALID_ARGUMENT, "the ring buffer of max_lag points per chain would exceed 48 GiB");
        // lags 1, 2, 3, 4, 6, 8, 12, 16, ... up to max_lag (MakeAutocorrelation.C:99-101 also samples the lags)
        e->diagLags.clear();
        for (int lag = 1; lag <= max_lag;) {
            e->diagLags.push_back(lag);
            if (lag < 4) ++lag;
            else if ((lag & (lag - 1)) == 0) lag += lag / 2;
            else lag = (lag / 3) * 4;
        }
        e->diagDepth = max_lag;
        if (smcmc_engine::poolAccSmem(e->n()) > 48 * 1024)
            CUDA_CHECK(cudaFuncSetAttribute(kPoolAccumulate, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)smcmc_engine::poolAccSmem(e->n())));
        e->diagPooled.reserve(e->poolStatCount());
        e->diagS1.reserve(En);
        e->diagS2.reserve(En);
        e->diagChainCount.reserve(e->E());
        if (max_lag > 0) {
            e->diagRing.reserve((size_t)max_lag * En);
            e->diagLagProd.reserve(e->diagLags.size() * e->n());
            e->diagLagCount.reserve(e->diagLags.size());
            e->diagLagsDev.reserve(e->diagLags.size());
            CUDA_CHECK(cudaMemcpy(e->diagLagsDev.get(), e->diagLags.data(), e->diagLags.size() * sizeof(int),
                                  cudaMemcpyHostToDevice));
        }
        e->diagReset();
        e->diagOn = true;
    });
}

int smcmc_diag_reset(smcmc_engine* e) {
    return guarded(e, [&]() {
        if (!e->diagOn) throw Error(SMCMC_ERR_LOGIC, "diagnostics are not enabled (smcmc_diag_enable)");
        e->diagReset();
    });
}

int smcmc_diag_lag_count(smcmc_engine* e, int32_t* nlags) {
    return guarded(e, [&]() {
        if (!nlags) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null output");
        *nlags = (int32_t)e->diagLags.size();
    });
}

int smcmc_diag_get(smcmc_engine* e, const smcmc_diag_result* out) {
    return guarded(e, [&]() {
        if (!e->diagOn) throw Error(SMCMC_ERR_LOGIC, "diagnostics are not enabled (smcmc_diag_enable)");
        if (!out) throw Error(SMCMC_ERR_INVALID_ARGUMENT, "null result");
        const size_t E = e->E(), n = e->n(), nl = e->diagLags.size();
        CUDA_CHECK(cudaStreamSynchronize(e->stream));
        std::vector<double> pooled(e->poolStatCount()), s1(E * n), s2(E * n), cc(E), lp(nl * n), lc(nl);
        CUDA_CHECK(cudaMemcpy(pooled.data(), e->diagPooled.get(), pooled.size() * 8, cudaMemcpyDeviceToHost));
        CUDA_CHECK(cudaMemcpy(s1.data(), e->diagS1.get(), s1.size() * 8, cudaMemcpyDeviceToHost));
        CUDA_CHECK(cudaMemcpy(s2.data(), e->diagS2.get(), s2.size() * 8, cudaMemcpyDeviceToHost));
        CUDA_CHECK(cudaMemcpy(cc.data(), e->diagChainCount.get(), cc.size() * 8, cudaMemcpyDeviceToHost));
        if (nl) {
            CUDA_CHECK(cudaMemcpy(lp.data(), e->diagLagProd.get(), lp.size() * 8, cudaMemcpyDeviceToHost));
            CUDA_CHECK(cudaMemcpy(lc.data(), e->diagLagCount.get(), lc.size() * 8, cudaMemcpyDeviceToHost));
        }
        const double count = pooled[0];
        if (out->samples) *out->samples = (int64_t)count;
        if (out->steps) *out->steps = (int64_t)e->diagFills;
        std::vector<double> mean(n, 0.0), var(n, 0.0);
        for (size_t i = 0; i < n; ++i) {                                   // MakeCovariance.C:76-83
            mean[i] = pooled[1 + i] / count;
            var[i] = pooled[1 + n + i * (i + 1) / 2 + i] / count - mean[i] * mean[i];
        }
        if (out->mean) std::copy(mean.begin(), mean.end(), out->mean);
        if (out->covariance) {
            for (size_t i = 0; i < n; ++i)
                for (size_t j = 0; j < n; ++j) {
                    const size_t hi = std::max(i, j), lo = std::min(i, j);
                    out->covariance[i * n + j] = pooled[1 + n + hi * (hi + 1) / 2 + lo] / count - mean[i] * mean[j];
                }
        }
        if (out->rhat) {
            // Gelman-Rubin: W = mean within-chain variance, B/N = variance of the chain means
            const double N = (double)e->diagFills;
            for (size_t i = 0; i < n; ++i) {
                double W = 0.0, m1 = 0.0, m2 = 0.0;
                size_t M = 0;
                for (size_t c = 0; c < E; ++c) {
                    // only chains that ran at every accumulated step (a chain that sits at 0 runs too)
                    if (cc[c] != N) continue;
                    const double a = s1[c * n + i], b = s2[c * n + i];
                    const double cm = a / N;
                    W += (b - N * cm * cm) / (N - 1.0);
                    m1 += cm;
                    m2 += cm * cm;
                    ++M;
                }
                double r = std::numeric_limits<double>::quiet_NaN();
                if (M > 1 && N > 1.0) {
                    W /= (double)M;
                    const double grand = m1 / (double)M;
                    const double BoverN = (m2 - (double)M * grand * grand) / ((double)M - 1.0);
                    r = std::sqrt(((N - 1.0) / N * W + BoverN) / W);
                }
                out->rhat[i] = r;
            }
        }
        if (out->lags) std::copy(e->diagLags.begin(), e->diagLags.end(), out->lags);
        std::vector<double> rho(nl * n, 0.0);
        for (size_t l = 0; l < nl; ++l)
            for (size_t i = 0; i < n; ++i)                                 // MakeAutocorrelation.C:131-136
                rho[l * n + i] = (lp[l * n + i] / lc[l] - mean[i] * mean[i]) / var[i];
        if (out->autocorrelation) std::copy(rho.begin(), rho.end(), out->autocorrelation);
        if (out->tau || out->ess) {
            // integrated autocorrelation time tau = 1 + 2 sum_{k>=1} rho(k): rho is taken
            // piecewise linear between the sampled lags (rho(0) = 1) and the sum stops at
            // the first zero crossing
            for (size_t i = 0; i < n; ++i) {
                double S = 0.0, prevLag = 0.0, prevRho = 1.0;
                for (size_t l = 0; l < nl; ++l) {
                    if (!(lc[l] > 0.0)) break;
                    const double r = rho[l * n + i], lag = (double)e->diagLags[l];
                    const double w = lag - prevLag, m = (r - prevRho) / w;
                    if (r > 0.0) {
                        S += w * prevRho + m * w * (w + 1.0) / 2.0;
                        prevLag = lag;
                        prevRho = r;
                    } else {
                        const double k = std::floor(prevRho / (-m));
                        S += k * prevRho + m * k * (k + 1.0) / 2.0;
                        break;
                    }
                }
                const double tau = 1.0 + 2.0 * S;
                if (out->tau) out->tau[i] = tau;
                if (out->ess) out->ess[i] = count / tau;
            }
        }
    });
}

int smcmc_pair_kernel_stats(smcmc_engine* e, double* totalMs, int64_t* launches, int reset) {
    return guarded(e, [&]() {
        e->collectPairTimings();
        if (totalMs) *totalMs = e->pairMs;
        if (launches) *launches = e->pairLaunches;
        if (reset) {
            e->pairMs = 0.0;
            e->pairLaunches = 0;
        }
    });
}

}  // extern "C"

#include "engine_hmc.inl"
