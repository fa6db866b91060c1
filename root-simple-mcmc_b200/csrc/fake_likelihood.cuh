// fake_likelihood.cuh -- the event-loop likelihood of example/FakeLikelihood.H
// for many parameter points (chains) at once.
//
// Reference: FakeLikelihood::operator() (example/FakeLikelihood.H:47-81),
// FillHistograms (:188-216), SystematicCorrection::{InvariantMass,Separation,
// EventWeight,CorrectEvent} (example/SystematicCorrection.H:35-128).
//
// How the work is cut (DESIGN.md section 3):
//  * Everything that depends only on the EVENT (3 logs, one division) is
//    computed once when the sample is uploaded: PreparedEvent, 32 bytes.
//  * Everything that depends only on the CHAIN (5 exp, erf, 2 atan) is computed
//    once per likelihood evaluation: FakeChainParams.
//  * What is left per (chain, event) pair is one exp, 7 FP64 operations in the
//    reference's order, and a bin lookup.  The corrected mass itself is never
//    exponentiated: TH1's bin of exp(l) is found by comparing l with the
//    pre-image of the bin edges under the host's exp (gEdges), which is the
//    same decision as the reference's exp-then-FindBin.
//  * An event's weight takes one of four values per chain (signal/background x
//    decay tag), so the histograms are accumulated as exact INTEGER counts per
//    weight class and turned into the reference's sequentially-rounded bin
//    contents afterwards (seqsum.h).  Integer counts make the result
//    independent of event order, of the tiling and of the number of GPUs.
//  * Pair kernel: one CTA = 256 chains (one per thread) x one chunk of events
//    of a single weight class.  Event tiles are staged into shared memory by
//    TMA bulk copies (cp.async.bulk + mbarrier, double buffered) and every
//    thread reads them by broadcast; each thread owns a private column of
//    shared-memory counters, so no atomics and no bank conflicts.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "seqsum.h"
#include "smcmc_b200.h"
#include "smcmc_tma.cuh"

namespace smcmc {

// Per-event constants (example/SystematicCorrection.H:53-62).
struct __align__(32) PreparedEvent {
    double logSigma;   // (log m - log M0) / (log(M0+S0) - log M0)
    double dLog;       // log m - log M0
    double nomLog;     // log M0
    double sep;        // evt.Separation
};
static_assert(sizeof(PreparedEvent) == 32, "PreparedEvent is 32 bytes");

// Per-chain constants.
struct FakeChainParams {
    double skewc;      // 0.3*erf(p[kMassSkew]/10)              :68
    double width;      // exp(p[kMassWidth]/10)                 :65
    double scale;      // p[kMassScale]/10                      :64
    double sepScale[2];// exp((0+p[5|6])/10)  signal, background :42-45
    double weight[4];  // [signal, signal&tag, background, background&tag] :81-117
};

// Weight classes and the layout of the count table.
//   class 0: signal, MuDk==0     -> slots [  0,100)  Close bins, Separated bins
//   class 1: signal, MuDk>0      -> slots [100,150)  DecayTag bins
//   class 2: background, MuDk==0 -> slots [150,250)
//   class 3: background, MuDk>0  -> slots [250,300)
//   class 4: data-typed (Type<0) -> slots [300,450)  Close, Separated, DecayTag
// counts[slot][point] (point fastest) are uint32.
constexpr int kFakeClasses = 4;
constexpr int kFakeSlots = 450;
__host__ __device__ constexpr int fakeClassSlotBase(int cls) {
    return cls == 0 ? 0 : cls == 1 ? 100 : cls == 2 ? 150 : cls == 3 ? 250 : 300;
}
constexpr int kIrregularClass = 5;   // events the fast path cannot take

constexpr int kPairThreads = 256;    // chains per CTA
constexpr int kPairTile = 128;       // events per shared-memory tile
constexpr int kPairChunk = 8192;     // most events per CTA work item
constexpr int kPairCounterRows = 100;
// Private shared-memory counters are 16 bits wide (a chunk has fewer than 65536
// events), two chains per 32-bit word: four CTAs fit one SM.
#ifndef SMCMC_PAIR_CTAS
#define SMCMC_PAIR_CTAS 4
#endif
#ifndef SMCMC_PAIR_EXPERIMENT
#define SMCMC_PAIR_EXPERIMENT 0
#endif
#ifndef SMCMC_PAIR_UNROLL
#define SMCMC_PAIR_UNROLL 2
#endif
constexpr int kPairCtasPerSm = SMCMC_PAIR_CTAS;
constexpr int kPairUnroll = SMCMC_PAIR_UNROLL;    // groups of four events in flight per thread
static_assert(kPairChunk < (1 << 16), "a chunk must not overflow a counter");

// Pre-images of the 50 bin edges under the host's exp, and of the cut at 500:
//   bin (1-based) of exp(l) is 1 + #{k in 1..49 : l >= gEdges[k]},
//   the event is dropped when !(l < gEdges[50]).
__constant__ double gEdges[52];
// tan(M_PI*(trueFakes-0.5)), tan(M_PI*(trueEfficiency-0.5)), M_PI: host values.
__constant__ double gFakeConst[4];

// ---------------------------------------------------------------------------
// Upload-time preparation.
// ---------------------------------------------------------------------------
__device__ __forceinline__ int classifyEvent(const smcmc_event& e, PreparedEvent& p) {
    double nomLog = log(e.TrueMass);                                   // :57
    double nomLogSigma = log(__dadd_rn(e.TrueMass, e.TrueMassSigma));  // :58
    nomLogSigma = __dsub_rn(nomLogSigma, nomLog);                      // :59
    double logMass = log(e.Mass);                                      // :61
    double d = __dsub_rn(logMass, nomLog);
    p.dLog = d;
    p.logSigma = __ddiv_rn(d, nomLogSigma);                            // :62
    p.nomLog = nomLog;
    p.sep = e.Separation;
    bool regular = e.Type >= 0 && isfinite(p.dLog) && isfinite(p.logSigma) &&
                   isfinite(p.nomLog) && isfinite(p.sep) && p.sep >= 0.0 &&
                   fabs(p.nomLog) <= 11.0 &&    // |nomLog*log2(e)| <= 16: filter guard
                   fabs(p.logSigma) <= 36.0;    // |logSigma*scl2| <= 16 for every chain: filter guard
    if (!regular) return kIrregularClass;
    return (e.Type == 0 ? 0 : 2) + (e.MuDk > 0 ? 1 : 0);
}

// Mass bands of the layout: events of a class are grouped by observed Mass around the cut at 500, so
// that the events above the cut for a whole box of chains fill whole tiles (the tile skip of
// pairChunk).  Band b holds edge[b-1] <= Mass < edge[b] (massBand); the edges were chosen with
// scripts/skip_fraction.py.  Bands from kFirstCandidateBand on are the ones whose tiles the pair
// kernel tests; the layout is only a heuristic, no count depends on it.
constexpr int kMassBands = 6;
constexpr int kFirstCandidateBand = 1;
constexpr int kBandSlots = 8;                // per class in the upload's counters (kFakeCountClasses)
__device__ __forceinline__ int massBand(double mass) {
    const double edge[kMassBands - 1] = {450.0, 550.0, 600.0, 700.0, 900.0};
    int b = 0;
#pragma unroll
    for (int k = 0; k < kMassBands - 1; ++k) b += mass >= edge[k] ? 1 : 0;
    return b;
}
__device__ __forceinline__ int eventBand(const smcmc_event& e, int cls) {
    return cls == kIrregularClass ? 0 : massBand(e.Mass);
}

// counts[cls * kBandSlots + band]: events per class and mass band.
__global__ void kFakeCountClasses(const smcmc_event* __restrict__ ev, int64_t n,
                                  unsigned long long* counts, int forceGeneric) {
    constexpr int kSlots = 8 * kBandSlots;
    __shared__ unsigned int local[kSlots];
    if (threadIdx.x < kSlots) local[threadIdx.x] = 0;
    __syncthreads();
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        PreparedEvent p;
        int cls = forceGeneric ? kIrregularClass : classifyEvent(ev[i], p);
        atomicAdd(&local[cls * kBandSlots + eventBand(ev[i], cls)], 1u);
    }
    __syncthreads();
    if (threadIdx.x < kSlots && local[threadIdx.x])
        atomicAdd(&counts[threadIdx.x], (unsigned long long)local[threadIdx.x]);
}

// Re-layout at upload.  Events are ordered by (class, mass band, secondary key): inside a class the
// order does not matter for the counts.  The bands put the events that are above the mass cut for
// a whole box of chains together (the tile skip).  Inside a band, the untagged classes are ordered
// by ascending separation, which makes most of their tiles lie entirely on one side of every chain's
// separation cut, so that the pair kernel can skip the per-pair test there (pairChunk); the tagged
// classes have no separation test and are ordered by observed mass.  kFakeSortKeys writes the
// 64-bit sort keys (class << 36 | band << 32 | secondary), the host sorts (key, index) with a device
// radix sort over bits 0..38, kFakeGather fills the class segments.
constexpr int kSortKeyBits = 39;
struct FilterTile;
__device__ __forceinline__ void storeFilterEvent(FilterTile* tiles, int64_t idx, const PreparedEvent& p);

__global__ void kFakeSortKeys(const smcmc_event* __restrict__ ev, int64_t n, unsigned long long* keys,
                              unsigned int* index, int forceGeneric) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    PreparedEvent p;
    const int cls = forceGeneric ? kIrregularClass : classifyEvent(ev[i], p);
    unsigned int low = 0;                     // >= 0: bit order = value order
    if (cls == 0 || cls == 2) low = __float_as_uint(fabsf(__double2float_rn(p.sep)));
    else if (cls == 1 || cls == 3) low = __float_as_uint(fabsf(__double2float_rn(ev[i].Mass)));
    keys[i] = ((unsigned long long)cls << 36) | ((unsigned long long)eventBand(ev[i], cls) << 32) | low;
    index[i] = (unsigned int)i;
}

// sortedStart[c] = position of the first event of class c in the sorted order.
__global__ void kFakeGather(const smcmc_event* __restrict__ ev, int64_t n, const unsigned long long* __restrict__ keys,
                            const unsigned int* __restrict__ index, const int64_t* __restrict__ sortedStart,
                            const int64_t* __restrict__ classBase, PreparedEvent* prepared, FilterTile* filter,
                            smcmc_event* irregular) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int cls = (int)(keys[i] >> 36);
    const int64_t rank = i - sortedStart[cls];
    const smcmc_event e = ev[index[i]];
    if (cls == kIrregularClass) {
        irregular[rank] = e;
        return;
    }
    PreparedEvent p;
    classifyEvent(e, p);
    prepared[classBase[cls] + rank] = p;
    storeFilterEvent(filter, classBase[cls] + rank, p);
}

// ---------------------------------------------------------------------------
// Per-evaluation chain constants.
// ---------------------------------------------------------------------------
struct FilterChain;
__device__ __forceinline__ void storeFilterChain(FilterChain* dst, int c, const FakeChainParams& cp, int exactOnly);

// variant 0: example/SystematicCorrection.H; variant 1: example2/SystematicCorrection.H
// (:75-117), whose EventWeight has neither the exp(p/10) event-count factors nor
// the exposure ratio (the counts are applied by the renormalisation in kFake2Finish).
__device__ __forceinline__ void fakePairGeneric(const smcmc_event& e, const double* __restrict__ p, int point,
                                                uint32_t* counts, int blockPoints);
__global__ void kFakePrepareChains(const double* __restrict__ x, int m, int dim,
                                   double exposure, FakeChainParams* out, FilterChain* fout,
                                   int exactOnly, int variant, uint32_t* zero = nullptr, int zeroWords = 0,
                                   const smcmc_event* __restrict__ irregular = nullptr, int64_t irregularCount = 0,
                                   int blockPoints = 0) {
    // Few points (the streaming regime, ONE block): the small count table is cleared here instead of
    // by a memset node of its own, and the handful of events the tiles cannot hold (data-typed,
    // non-finite ...) are counted by the threads that have no chain to prepare -- the per-pair
    // transcription of the reference formula, concurrent with the chain constants below.
    if (zero) {
        for (int k = threadIdx.x; k < zeroWords; k += blockDim.x) zero[k] = 0u;
        __syncthreads();
        const int64_t pairs = irregularCount * m;
        for (int64_t idx = (int64_t)blockDim.x - 1 - threadIdx.x; idx < pairs; idx += blockDim.x) {
            const int point = (int)(idx % m);
            fakePairGeneric(irregular[idx / m], x + (size_t)point * dim, point, zero, blockPoints);
        }
    }
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= m) return;
    const double* p = x + (size_t)c * dim;
    FakeChainParams cp;
    cp.scale = __ddiv_rn(p[2], 10.0);                                  // :64
    cp.width = exp(__ddiv_rn(p[3], 10.0));                             // :65
    cp.skewc = __dmul_rn(0.3, erf(__ddiv_rn(p[4], 10.0)));             // :68
    cp.sepScale[0] = exp(__ddiv_rn(__dadd_rn(0.0, p[5]), 10.0));       // :41-45
    cp.sepScale[1] = exp(__ddiv_rn(__dadd_rn(0.0, p[6]), 10.0));
    const double pi = gFakeConst[2];
    double wSig = __dmul_rn(1.0, exp(__ddiv_rn(p[0], 10.0)));          // :88
    double wBkg = __dmul_rn(1.0, exp(__ddiv_rn(p[1], 10.0)));          // :89
    const double trueFakes = 0.05;                                     // :94-97
    double fakes = __dadd_rn(gFakeConst[0], p[7]);
    fakes = __dadd_rn(__ddiv_rn(atan(fakes), pi), 0.5);
    const double trueEff = 0.5;                                        // :106-109
    double eff = __dadd_rn(gFakeConst[1], p[8]);
    eff = __dadd_rn(__ddiv_rn(atan(eff), pi), 0.5);
    double sigTag = __dmul_rn(wSig, __ddiv_rn(fakes, trueFakes));                                   // :100
    double sigNo = __dmul_rn(wSig, __ddiv_rn(__dsub_rn(1.0, fakes), __dsub_rn(1.0, trueFakes)));    // :101
    double bkgTag = __dmul_rn(wBkg, __ddiv_rn(eff, trueEff));                                       // :112
    double bkgNo = __dmul_rn(wBkg, __ddiv_rn(__dsub_rn(1.0, eff), __dsub_rn(1.0, trueEff)));        // :113
    if (variant == 0) {
        cp.weight[0] = __dmul_rn(sigNo, exposure);                     // :116
        cp.weight[1] = __dmul_rn(sigTag, exposure);
        cp.weight[2] = __dmul_rn(bkgNo, exposure);
        cp.weight[3] = __dmul_rn(bkgTag, exposure);
    } else {
        // weight = 1.0; weight *= ratio  (example2/SystematicCorrection.H:76,98-99,110-111)
        cp.weight[0] = __dmul_rn(1.0, __ddiv_rn(__dsub_rn(1.0, fakes), __dsub_rn(1.0, trueFakes)));
        cp.weight[1] = __dmul_rn(1.0, __ddiv_rn(fakes, trueFakes));
        cp.weight[2] = __dmul_rn(1.0, __ddiv_rn(__dsub_rn(1.0, eff), __dsub_rn(1.0, trueEff)));
        cp.weight[3] = __dmul_rn(1.0, __ddiv_rn(eff, trueEff));
    }
    out[c] = cp;
    storeFilterChain(fout, c, cp, exactOnly);
}

// ---------------------------------------------------------------------------
// Bin lookup (exact).
// ---------------------------------------------------------------------------
// 0-based bin of a corrected log-mass, or 50 when the event is cut
// (FakeLikelihood.H:203-204 and the TH1 overflow bin).  NaN is cut.
__device__ __forceinline__ int exactBin(double lm, int guess) {
    if (!(lm < gEdges[50])) return 50;
    int k = min(max(guess, 0), 49);
    while (k > 0 && lm < gEdges[k]) --k;
    while (k < 49 && lm >= gEdges[k + 1]) ++k;
    return k;
}

// The reference's arithmetic for one (chain, event) pair in FP64, operation
// for operation (SystematicCorrection.H:69-74, :45-47; FakeLikelihood.H:
// 203-214).  Returns the counter row (bin, +50 for the Separated histogram of
// untagged events) or -1 when the event is cut.
__device__ __forceinline__ int exactDecide(const PreparedEvent& ev, const FakeChainParams& cp,
                                           int cls) {
    double skew = exp(__dmul_rn(ev.logSigma, cp.skewc));
    double lm = __dadd_rn(ev.nomLog, __dmul_rn(ev.dLog, skew));
    lm = __dadd_rn(ev.nomLog, __dmul_rn(__dsub_rn(lm, ev.nomLog), cp.width));
    lm = __dadd_rn(lm, cp.scale);
    int guess = (int)(__expf((float)lm) * 0.1f);      // any guess is corrected below
    int bin = exactBin(lm, guess);                    // mass = exp(lm); TH1 bin of mass
    if (bin >= 50) return -1;
    if (!(cls & 1)) {
        double sep = __dmul_rn(ev.sep, cp.sepScale[cls >> 1]);
        if (!(sep < 100.0)) bin += 50;
    }
    return bin;
}

// ---------------------------------------------------------------------------
// The FP32 interval filter.
//
// Only a DISCRETE decision is needed per pair: which counter row, or none.
// The filter evaluates q = mass/10 in FP32 together with a rigorous bound m on
// its relative error and accepts the FP32 decision only when q(1-m) and q(1+m)
// have the same integer part (and the scaled separation is farther than its
// bound from 100).  Everything else is "unsure" and is re-evaluated with
// exactDecide.  The filter therefore never changes a count; it only decides
// which pairs need FP64.
//
// Arithmetic (log2 domain; K = 2^c2 with c2 = scale*log2(e) - log2(10) is a per-chain constant
// that never meets the per-pair exponent: it multiplies the error-bound factors instead):
//   x2 = ls*scl2;  t = d*ex2(x2);  z = fma(t, w2, nl2);  q' = ex2(z);      q = K q'
//   A = fma(|t|, aT, a0) = K(1+m),  B = 2K - A = K(1-m)     (m = m0 + slopeT|t|, the bound below)
//   hi = RZ(fma(q', A, 1.5*2^23)),  lo = RZ(fma(q', B, 1.5*2^23))
// The products q'A and q'B are exact inside the FMAs and the round-toward-zero sum with 1.5*2^23
// is their integer part on the float grid: hi = floor(q(1+m)), lo = floor(q(1-m)), one instruction
// each, no second rounding.
//
// Error bound (u = 2^-24; inputs are correctly rounded to FP32):
//   x2 = ls*scl2             rel. error <= 3u
//   skew = ex2.approx(x2)    rel. error <= 4u + ln2*3u|x2|          (2 ulp unit)
//   t = d*skew               rel. error <= (6 + 2.08|x2|)u
//   z = fma(t, w2, nl2)      abs. error <= u[(8+2.08|x2|)|t w2| + 2|nl2|]
//   q' = ex2.approx(z)       rel. error <= 4u + ln2*abs.err(z)
//   K, A as floats           rel. error <= u/2 (K), u (A: one FMA rounding on [K, 2K));
//                            B = 2K - A is exact (Sterbenz) while m <= 3
// |x2| <= 16 holds for every pair because |scl2| = |0.3 erf(.) log2 e| <= 0.4329
// and events with |logSigma| > 36 are kept out of the fast path at upload;
// |nl2| <= 16 is checked per event at upload as well.  With those guards
//   rel(q') <= u[4 + ln2 (2*16)] + u ln2 (8 + 2.08*16)|t w2| = u[26.2 + 28.6|t w2|],
// and the interval [q'B, q'A] holds the exact q when m >= rel(q') + 3u (K, A and 2K as floats):
//   m >= u[29.2 + 28.6|t w2|]  (first order; the second-order terms are below 1e-3 u).
// The code uses kFilterSafety = 1.5 times that (round 1 used 2 x u[48.4 + 2.78|c2| + 30.5|t w2|]: the
// c2 terms went with the addition, and every undecided pair costs an FP64 evaluation).
// Chains whose constants leave the range this analysis covers (|c2| > 24, |w2| > 2^24, anything
// non-finite) and SMCMC_FAKE_EXACT carry force = 1: every pair of theirs goes to FP64.
//
// Data layout.  Events of a class are stored in TILES of 128, structure of
// arrays inside a tile (FilterTile, 2 KB, one TMA bulk copy), and every class
// segment is padded to a whole number of tiles with records that can never be
// counted (nl2 = +inf).  A thread therefore reads four events' worth of one
// field with a single broadcast LDS.128, and the arithmetic runs on PAIRS of
// events with the packed FP32x2 instructions of sm_100 (FMUL2 / FFMA2 / FADD2:
// two roundings per issue slot, identical results to the scalar instructions).
// ---------------------------------------------------------------------------
struct __align__(16) FilterTile {
    float ls[kPairTile];     // logSigma
    float d[kPairTile];      // dLog
    float nl2[kPairTile];    // nomLog * log2(e)
    float sep[kPairTile];
};
static_assert(sizeof(FilterTile) == 16 * kPairTile, "FilterTile is 16 bytes per event");

constexpr double kFilterSafety = 1.5;
struct __align__(16) FilterChain {
    float scl2;      // skewc * log2(e)
    float w2;        // width * log2(e)
    float a0;        // K (1 + m0),  K = 2^(scale*log2(e) - log2(10)), m0 = constant part of the error bound of q
    float aT;        // K slopeT: the bound grows by slopeT * |d*skew|
    float twoK;      // 2 K
    float thr[2];    // 100 / separation scale: signal, background
    float thrEps[2]; // error bound of the comparison  sep <> thr
    uint32_t force;  // 1: the filter is not used for this chain (every pair in FP64)
    float cutZ;      // log2(500) - scale*log2(e), rounded up: the tile skip's threshold (tileAllCut)
    float pad_;
};
static_assert(sizeof(FilterChain) == 48, "FilterChain is 48 bytes");

__device__ __forceinline__ void storeFilterEvent(FilterTile* tiles, int64_t idx, const PreparedEvent& p) {
    FilterTile& t = tiles[idx / kPairTile];
    const int k = (int)(idx % kPairTile);
    t.ls[k] = __double2float_rn(p.logSigma);
    t.d[k] = __double2float_rn(p.dLog);
    t.nl2[k] = __double2float_rn(p.nomLog * 1.4426950408889634);
    t.sep[k] = __double2float_rn(p.sep);
}

// Padding records of one class segment [base+real, base+padded): q = 2^(+inf) is
// cut in FP32 and nomLog = +inf is cut in FP64, so they are never counted; their
// separation repeats the last real one so that a tile's first and last
// separation stay its minimum and maximum.
__global__ void kFakePadEvents(PreparedEvent* prepared, FilterTile* tiles, int64_t base, int64_t real, int64_t padded) {
    int64_t i = base + real + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= base + padded) return;
    const float inf = __int_as_float(0x7f800000);
    float sep = 0.f;
    if (real > 0) {
        const int64_t last = base + real - 1;
        sep = tiles[last / kPairTile].sep[last % kPairTile];
    }
    FilterTile& t = tiles[i / kPairTile];
    const int k = (int)(i % kPairTile);
    t.ls[k] = 0.f;
    t.d[k] = 0.f;
    t.nl2[k] = inf;
    t.sep[k] = sep;
    PreparedEvent p;
    p.logSigma = 0.0;
    p.dLog = 0.0;
    p.nomLog = (double)inf;
    p.sep = 0.0;
    prepared[i] = p;
}

// exactOnly (SMCMC_FAKE_EXACT=1): an infinite error bound makes every pair
// "unsure", i.e. the whole evaluation runs through the FP64 arithmetic.
__device__ __forceinline__ void storeFilterChain(FilterChain* dst, int c, const FakeChainParams& cp, int exactOnly) {
    const double log2e = 1.4426950408889634, log2ten = 3.3219280948873623;
    const double u = 5.9604645e-8;
    FilterChain f;
    f.scl2 = __double2float_rn(cp.skewc * log2e);
    const double w2 = cp.width * log2e;
    f.w2 = __double2float_rn(w2);
    const double c2 = cp.scale * log2e - log2ten;
    const double K = exp2(c2);
    const double m0 = kFilterSafety * u * 29.2;
    const double slopeT = kFilterSafety * u * 28.6 * fabs(w2);
    f.a0 = __double2float_ru(K * (1.0 + m0));
    f.aT = __double2float_ru(K * slopeT);
    f.twoK = __double2float_rn(2.0 * K);
    const bool covered = isfinite(cp.skewc) && fabs(w2) <= 16777216.0 && fabs(c2) <= 24.0;   // false for NaN
    f.force = (exactOnly || !covered) ? 1u : 0u;
    if (f.force) {
        // lo != hi (or NaN) for every pair: the kernels that decide pair by pair (kFakeStream,
        // kFakeVerifyFilter) need no flag
        f.a0 = __int_as_float(0x7f800000);
        f.aT = 0.f;
        f.twoK = 1.f;
        if (!covered) f.scl2 = f.w2 = 0.f;
    }
    for (int k = 0; k < 2; ++k) {
        const double thr = 100.0 / cp.sepScale[k];
        f.thr[k] = __double2float_rn(thr);
        f.thrEps[k] = __double2float_ru(8.0 * u * fabs(thr));
    }
    f.cutZ = __double2float_ru(8.965784284662087 - cp.scale * log2e);     // log2(500)
    f.pad_ = 0.f;
    dst[c] = f;
}

__device__ __forceinline__ float fastEx2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ uint32_t smemAddr(const void* p);

// The filter on two events at once.  For each half: lo = RZ(q(1-m) + 1.5*2^23)
// and hi = RZ(q(1+m) + 1.5*2^23) sit on the integer grid, so the pair is
// decided ("sure") when lo == hi as FLOATS (NaN is never sure; +inf is, and is
// cut), and then counted in row floor(q) = bits(lo) - 0x4b400000 when that is
// below 50 (mass < 500).  ds = sep - 100/scale for the separation test.
constexpr unsigned kFloorMagicBits = 0x4b400000u;
constexpr int kFilterCutRow = 50;

struct FilterPair {
    float2 lo, hi, ds;
};

template <bool TAGGED>
__device__ __forceinline__ FilterPair filterCore2(float2 ls, float2 d, float2 nl2, float2 sep,
                                                  const FilterChain& fc, float thr) {
    const float2 x2 = __fmul2_rn(ls, make_float2(fc.scl2, fc.scl2));
    const float2 t = __fmul2_rn(d, make_float2(fastEx2(x2.x), fastEx2(x2.y)));
    const float2 z = __ffma2_rn(t, make_float2(fc.w2, fc.w2), nl2);
    const float2 q = make_float2(fastEx2(z.x), fastEx2(z.y));                       // q' = q / K
    const float2 a = make_float2(fmaf(fabsf(t.x), fc.aT, fc.a0), fmaf(fabsf(t.y), fc.aT, fc.a0));
    const float2 b = __fadd2_rn(make_float2(fc.twoK, fc.twoK), make_float2(-a.x, -a.y));
    const float2 magic = make_float2(12582912.0f, 12582912.0f);
    FilterPair r;
    r.hi = __ffma2_rz(q, a, magic);
    r.lo = __ffma2_rz(q, b, magic);
    r.ds = TAGGED ? make_float2(0.f, 0.f) : __fadd2_rn(sep, make_float2(-thr, -thr));
    return r;
}

// The discrete decision of one half.
struct FilterDecision {
    bool sure;       // the FP32 decision is provably the FP64 decision
    bool counted;    // sure, and the event falls in a histogram bin
    unsigned bits;   // 0x4b400000 + floor(q)
    bool far;        // separation >= 100 (untagged classes only)
};
template <bool TAGGED>
__device__ __forceinline__ FilterDecision filterDecide(float lo, float hi, float ds, float thrEps) {
    FilterDecision r;
    r.sure = (lo == hi);
    r.far = false;
    if (!TAGGED) {
        r.sure = r.sure & (fabsf(ds) > thrEps);
        r.far = ds > 0.0f;
    }
    r.bits = __float_as_uint(lo);
    r.counted = r.sure & (r.bits < kFloorMagicBits + kFilterCutRow);
    return r;
}

// Counters.  A CTA holds 101 rows x 256 chains of 16-bit counters, packed two
// per 32-bit word (chains c and c+128 -> word c), and EVERY update is a shared-memory
// atomic add without a return value (RED): one instruction instead of a
// load/add/store chain, and the deferred FP64 pass may update any chain's
// column.  16 bits cannot overflow within a chunk (kPairChunk < 65536), so the
// low half never carries into the high half.
//
// Row layout: bins of the Close histogram (tagged classes: DecayTag) in rows 0..49 ascending,
// row 50 takes the events that are cut (mass >= 500), the Separated histogram in rows 100..51
// DESCENDING (bin b -> row 100 - b).  Both histograms reach the cut row by clamping the bin
// at 50: the address of an event is  min(bits, 0x4b400032) * (+-512) + constant,
// with no comparison, no select and no branch.
constexpr unsigned kPairRowBytes = (kPairThreads / 2) * sizeof(uint32_t);
static_assert(kPairRowBytes == 512, "row stride of the counter table");
constexpr int kPairCutRow = kFilterCutRow;
constexpr int kPairFarRow0 = 2 * kFilterCutRow;                  // row of Separated bin 0
__host__ __device__ constexpr int pairRowOfBin(int bin) {         // bin: 0..49 Close, 50..99 Separated
    return bin < kFilterCutRow ? bin : kPairFarRow0 - (bin - kFilterCutRow);
}

__device__ __forceinline__ void redShared(unsigned addr, unsigned value) {
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(value) : "memory");
}

// ---------------------------------------------------------------------------
// The pair kernel.
// ---------------------------------------------------------------------------
// The count table is cut into blocks of blockPoints consecutive points, each block a
// [kFakeSlots][blockPoints] array (point fastest).  One block (blockPoints = row length) is
// the plain [slot][point] table; with the events split over G GPUs block r is what rank r
// receives from the reduce-scatter and finishes (engine.cu, evaluateFake).
__device__ __forceinline__ size_t countIndex(int slot, int point, int blockPoints) {
    const int b = point / blockPoints;
    return ((size_t)b * kFakeSlots + slot) * (size_t)blockPoints + (size_t)(point - b * blockPoints);
}

struct PairLaunch {
    const PreparedEvent* events;     // FP64 records; class segments contiguous, padded to whole tiles
    const FilterTile* filterTiles;   // FP32 records, same order, 128 per tile
    int64_t classBase[kFakeClasses]; // first (padded) event index of each class, a multiple of kPairTile
    int64_t classCount[kFakeClasses];// events of the class INCLUDING the padding of its last tile
    int64_t classReal[kFakeClasses]; // events of the class without the padding
    int64_t bandStart[kFakeClasses][kMassBands];   // first event of each mass band, relative to classBase
    int skipTiles;                   // the tile skip is on (off: SMCMC_FAKE_NO_SKIP)
    int chunkBase[kFakeClasses + 1]; // prefix sum of chunks per class
    int chunkEvents;                 // events per work item (multiple of kPairTile, <= kPairChunk)
    const FakeChainParams* chains;
    const FilterChain* filterChains;
    int numPoints;                   // chains (parameter points) to evaluate
    int pointStride;                 // points the count table has room for
    int blockPoints;                 // points per block of the count table (countIndex); == pointStride: one block
    uint32_t* counts;                // [block][kFakeSlots][blockPoints]
    unsigned long long* stats;       // optional: [0] unsure pairs, [1] pairs in skipped tiles
};

// Undecided pairs are not evaluated where they are found (one lane in FP64
// while 31 wait): a lane appends them to its WARP's queue in shared memory, and the warp works
// its queue off by itself, one pair per lane, at the end of a tile once kPairDrainAt pairs
// have gathered (and at the end of the chunk).  No CTA-wide barrier is involved; pairs that do not
// fit are evaluated in place.
constexpr int kPairWarps = kPairThreads / 32;
constexpr int kPairQueueCap = 30;        // per warp
constexpr int kPairDrainAt = 16;
struct PairQueue {
    unsigned done[2];                    // warps that have finished the tile in each buffer
    unsigned unsure;                     // pairs that went to FP64 (statistics)
    int cls;                             // what exactCount needs, for the lanes that find their queue full
    const PreparedEvent* chunkEvents;
    const FakeChainParams* chains;       // of the CTA's first chain
    unsigned countersAddr;
    unsigned skipped;                    // pairs in tiles skipped by the warps (statistics)
    unsigned count[kPairWarps];
    unsigned entry[kPairWarps][kPairQueueCap];   // (event index in chunk) << 8 | chain index in CTA
};

constexpr size_t kPairSmemTiles = 2 * sizeof(FilterTile);
constexpr size_t kPairSmemCounters = (size_t)(kPairCounterRows + 1) * kPairRowBytes;
constexpr size_t kPairSmemBytes = kPairSmemTiles + 64 + kPairSmemCounters + sizeof(PairQueue);
static_assert(kPairCtasPerSm * (kPairSmemBytes + 1024) <= 232448, "resident CTAs per SM");

// FP64 evaluation of one undecided pair and its count.
__device__ __noinline__ void exactCount(const PreparedEvent* ev, const FakeChainParams* cp, int cls,
                                        unsigned countersAddr, int chain) {
    const int bin = exactDecide(*ev, *cp, cls);
    if (bin >= 0)
        redShared(countersAddr + (unsigned)pairRowOfBin(bin) * kPairRowBytes + (unsigned)(chain & (kPairThreads / 2 - 1)) * 4u,
                  (chain >= kPairThreads / 2) ? 65536u : 1u);
}

// The address arithmetic of one tile for one thread: counter of bin b = b * mul + adj for the
// bits b of a float on the 1.5*2^23 grid (0x4b400000 + integer part).
struct PairRows {
    unsigned mul, adj;         // the tile's histogram (Close / DecayTag ascending, or Separated descending)
    unsigned farMul, farAdj;   // the Separated histogram (tiles that test every pair)
};

// acc |= a ^ b: one LOP3 (an explicit lop3.b32 here crashes ptxas 12.9 in this kernel; tileLoop keeps
// the compiler from turning the accumulation into compares instead)
__device__ __forceinline__ void orXor(unsigned& acc, unsigned a, unsigned b) {
    acc |= a ^ b;
}

// Count one event PROVISIONALLY in the row of floor(q(1+m)): VIMNMX, IMAD, ATOMS.  Whether the
// decision stands is not looked at here: `acc` collects hi ^ lo over a group of four events
// (one LOP3 each), and a group with a non-zero acc is revisited by queueUnsure, which takes the
// provisional count of the undecided events back and queues them for FP64.
__device__ __forceinline__ void countFast(float lo, float hi, unsigned mul, unsigned adj, unsigned addValue, unsigned& acc) {
    const unsigned h = __float_as_uint(hi);
#if SMCMC_PAIR_EXPERIMENT == 1 || SMCMC_PAIR_EXPERIMENT == 3          // timing experiment (wrong counts): no atomic at all
    acc += min(h, kFloorMagicBits + kFilterCutRow) * mul + adj == 12345u ? 2u : 0u;
#elif SMCMC_PAIR_EXPERIMENT == 2        // timing experiment (wrong counts): the atomic predicated off
    const unsigned a = min(h, kFloorMagicBits + kFilterCutRow) * mul + adj;
    if (h == 0x4b400000u + 77u) redShared(a, addValue);
#else
    redShared(min(h, kFloorMagicBits + kFilterCutRow) * mul + adj, addValue);
#endif
    orXor(acc, h, __float_as_uint(lo));
}
// ... in a tile that straddles the separation cut of some chain: far events go to the Separated
// rows, and a separation within its error bound of the cut makes the event undecided as well.
__device__ __forceinline__ void countFastSep(float lo, float hi, float ds, float thrEps, const PairRows& rows,
                                             unsigned addValue, unsigned& acc) {
    const unsigned h = __float_as_uint(hi);
    const unsigned b = min(h, kFloorMagicBits + kFilterCutRow);
    const bool far = ds > 0.0f;
    redShared(far ? b * rows.farMul + rows.farAdj : b * rows.mul + rows.adj, addValue);
    orXor(acc, h, __float_as_uint(lo));
    if (!(fabsf(ds) > thrEps)) acc |= 1u;
}

// The rare path, out of line: queue one undecided pair of this lane (or evaluate it on the spot
// when the warp's queue is full).
__device__ __noinline__ void pushUnsure(PairQueue* queue, int eventInChunk) {
    const int tid = threadIdx.x;
    atomicAdd(&queue->unsure, 1u);
    const unsigned slot = atomicAdd(&queue->count[tid >> 5], 1u);
    if (slot < (unsigned)kPairQueueCap) queue->entry[tid >> 5][slot] = ((unsigned)eventInChunk << 8) | (unsigned)tid;
    else exactCount(queue->chunkEvents + eventInChunk, queue->chains + tid, queue->cls, queue->countersAddr, tid);
}
// One warp works its queue off: one pair per lane.
__device__ __noinline__ void drainWarpQueue(PairQueue* queue) {
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncwarp();
    const unsigned queued = min(queue->count[w], (unsigned)kPairQueueCap);
    if ((unsigned)lane < queued) {
        const unsigned e = queue->entry[w][lane];
        const int chain = (int)(e & 255u);
        exactCount(queue->chunkEvents + (e >> 8), queue->chains + chain, queue->cls, queue->countersAddr, chain);
    }
    __syncwarp();
    if (lane == 0) queue->count[w] = 0;
    __syncwarp();
}

// An iteration (eight events) of a tile held an undecided pair of this lane, or the lane's chain
// does not use the filter: take the provisional counts of the undecided events back and queue
// them for FP64.  The values are the ones the iteration has just computed -- nothing is
// evaluated again.
struct Settle8 {
    float lo[8], hi[8], ds[8];
};
template <bool NOSEP>
__device__ __forceinline__ void settleUnsure(const Settle8& v, float thrEps, const PairRows& rows,
                                             unsigned addValue, unsigned forceBit, PairQueue* queue, int event0) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const unsigned h = __float_as_uint(v.hi[k]);
        bool unsure = ((h ^ __float_as_uint(v.lo[k])) | forceBit) != 0u;
        if (!NOSEP && !(fabsf(v.ds[k]) > thrEps)) unsure = true;
        if (!unsure) continue;
        if (h < kFloorMagicBits + kFilterCutRow) {            // it was counted: take that back
            const bool far = !NOSEP && v.ds[k] > 0.0f;
            redShared(far ? h * rows.farMul + rows.farAdj : h * rows.mul + rows.adj, 0u - addValue);
        }
        pushUnsure(queue, event0 + k);
    }
}

// One tile of 128 events for one chain: eight events per iteration, four packed
// pairs whose dependency chains (LDS -> MUFU -> MUFU -> RED) overlap.
// NOSEP: no separation test (tagged classes, and tiles of the untagged classes
// that lie on one side of the cut for every chain of the CTA).
template <bool NOSEP>
__device__ __forceinline__ void tileLoop(const FilterTile* tile, const FilterChain& fc, float thr, float thrEps,
                                         const PairRows& rows, unsigned addValue, unsigned forceBit,
                                         PairQueue* queue, int tileBase) {
    const float4* ls4 = reinterpret_cast<const float4*>(tile->ls);
    const float4* d4 = reinterpret_cast<const float4*>(tile->d);
    const float4* nl4 = reinterpret_cast<const float4*>(tile->nl2);
    const float4* sp4 = reinterpret_cast<const float4*>(tile->sep);
#pragma unroll 1
    for (int g = 0; g < kPairTile / 4; g += 2) {
        FilterPair f[4];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
#if SMCMC_PAIR_EXPERIMENT == 3          // timing experiment (wrong counts): no shared-memory loads either
            const float gf = __int_as_float(0x3f800000 + ((g + h) << 12));
            const float4 ls = make_float4(gf, gf + 0.25f, gf + 0.5f, gf + 0.75f);
            const float4 d = make_float4(gf - 1.f, gf - 1.25f, gf - 1.5f, gf - 1.75f);
            const float4 nl = make_float4(gf + 1.f, gf + 1.25f, gf + 1.5f, gf + 1.75f);
#else
            const float4 ls = ls4[g + h], d = d4[g + h], nl = nl4[g + h];
#endif
            float4 sp = make_float4(0.f, 0.f, 0.f, 0.f);
            if (!NOSEP) sp = sp4[g + h];
            f[2 * h] = filterCore2<NOSEP>(make_float2(ls.x, ls.y), make_float2(d.x, d.y),
                                          make_float2(nl.x, nl.y), make_float2(sp.x, sp.y), fc, thr);
            f[2 * h + 1] = filterCore2<NOSEP>(make_float2(ls.z, ls.w), make_float2(d.z, d.w),
                                              make_float2(nl.z, nl.w), make_float2(sp.z, sp.w), fc, thr);
        }
        unsigned acc = forceBit;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (NOSEP) {
                countFast(f[k].lo.x, f[k].hi.x, rows.mul, rows.adj, addValue, acc);
                countFast(f[k].lo.y, f[k].hi.y, rows.mul, rows.adj, addValue, acc);
            } else {
                countFastSep(f[k].lo.x, f[k].hi.x, f[k].ds.x, thrEps, rows, addValue, acc);
                countFastSep(f[k].lo.y, f[k].hi.y, f[k].ds.y, thrEps, rows, addValue, acc);
            }
        }
        asm volatile("" : "+r"(acc));           // keep acc an integer (one LOP3 per event), not eight compares
        if (acc != 0u) {
            Settle8 v;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                v.lo[2 * k] = f[k].lo.x; v.lo[2 * k + 1] = f[k].lo.y;
                v.hi[2 * k] = f[k].hi.x; v.hi[2 * k + 1] = f[k].hi.y;
                v.ds[2 * k] = f[k].ds.x; v.ds[2 * k + 1] = f[k].ds.y;
            }
            settleUnsure<NOSEP>(v, thrEps, rows, addValue, forceBit, queue, tileBase + g * 4);
        }
    }
}

// ---------------------------------------------------------------------------
// The tile skip.
//
// Events above the mass cut (exactDecide returns -1: bin 50) produce nothing, and whether an event
// is cut depends on the chain only through scale, width and skewc:
//   lm = nomLog + width * dLog * exp(logSigma * skewc) + scale,   cut when lm >= gEdges[50] ~ log 500.
// width > 0, so over a BOX of chains (the min / max of each of the three over the live chains of a
// warp) the smallest lm of an event is reached at one corner: the least scale, and
//   dLog >= 0:  the least width and the least logSigma*skewc  (skewc low if logSigma >= 0, else high)
//   dLog <  0:  the largest width and the largest logSigma*skewc.
// In the log2 domain of the filter (ls, d, nl2 = the tile's FP32 records, s = skewc*log2(e),
// w = width*log2(e)) the test of one event at its corner is
//   x = ls*s;  t = d*ex2(x);  z = fma(t, w, nl2);   cut for the whole box when  z - err >= cutZ,
// cutZ = log2(500) - scale*log2(e) at the least scale, rounded up (FilterChain::cutZ).
//
// Error bound (u = 2^-24; z_real = nl2 + w*d*2^(ls*s) in real numbers at the real corner):
//   ls, d, nl2, s, w as floats   rel. error <= u each (nl2, s, w: an FP64 product rounded once)
//                                 -- the box of the FP32 s and w may lie inside the box of the
//                                 chains' exact values by as much: the same u, counted here
//   x = ls*s                     rel. error <= 3u (two inputs, one rounding), |x| <= 16 (filter guards)
//   ex2.approx(x)                rel. error <= 4u + ln2*3u|x| <= (4 + 2.08|x|)u
//   t = d*ex2                    rel. error <= (6 + 2.08|x|)u
//   z = fma(t, w, nl2)           abs. error <= |t w|(7 + 2.08|x|)u + |nl2|u + |z|u
//                                           <= u[41.4|t w| + 2|nl2|] <= u[41.4|t w| + 32]   (|nl2| <= 16)
// exactDecide computes lm in FP64 in the reference's order ((nom + d*skew) - nom, times width, plus
// nom, plus scale; exp within 1 ulp): each step rounds at 2^-53 of numbers below |nomLog| + |lm| +
// |width d skew|, and gEdges[50], the host-exp pre-image of 500, lies within 2^-51 log 500 of log 500.
// Together (and the rounding of cutZ from FP64) that is below 2^-45 (|t w| + 32) in log2 units:
// far below one u, covered by the +1 below.  So the kernel skips only when
//   z >= cutZ + err,  err = kSkipSafety * u * (42 |t| wHi + 33)
// (wHi >= w; both the slope and the offset rounded up, the sum with an FMA rounding up).  Then
// z_real >= cutZ_exact at the corner, every chain of the box has lm >= log 500 beyond the FP64
// rounding, and exactDecide returns -1 for every pair of the tile: skipping it changes no count.
// A warp with a `force` chain (non-finite or out-of-range constants, SMCMC_FAKE_EXACT) never
// skips; lanes without a chain take no part in the box.  NaN in z fails the comparison.
// ---------------------------------------------------------------------------
constexpr double kSkipSafety = 2.0;
struct SkipBox {
    float sLo, sHi, wLo, wHi;   // skewc*log2(e), width*log2(e) over the live chains of the warp
    float slope, zCut;          // err = slope |t| + (zCut - cutZ): see above
    bool valid;                 // the warp may skip tiles
};

// Warp-collective: every lane of the warp calls it.
__device__ __forceinline__ SkipBox warpSkipBox(const FilterChain& fc, bool live, bool enabled) {
    const float inf = __int_as_float(0x7f800000);
    SkipBox b;
    b.sLo = live ? fc.scl2 : inf;
    b.sHi = live ? fc.scl2 : -inf;
    b.wLo = live ? fc.w2 : inf;
    b.wHi = live ? fc.w2 : -inf;
    float cut = live ? fc.cutZ : -inf;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        b.sLo = fminf(b.sLo, __shfl_xor_sync(0xffffffffu, b.sLo, o));
        b.sHi = fmaxf(b.sHi, __shfl_xor_sync(0xffffffffu, b.sHi, o));
        b.wLo = fminf(b.wLo, __shfl_xor_sync(0xffffffffu, b.wLo, o));
        b.wHi = fmaxf(b.wHi, __shfl_xor_sync(0xffffffffu, b.wHi, o));
        cut = fmaxf(cut, __shfl_xor_sync(0xffffffffu, cut, o));
    }
    const double u = 5.9604644775390625e-8;
    b.slope = __double2float_ru(kSkipSafety * u * 42.0 * (double)b.wHi);
    b.zCut = __double2float_ru((double)cut + kSkipSafety * u * 33.0);
    // (fminf / fmaxf drop NaN: a NaN constant sets force, and force turns the skip off)
    const bool finite = isfinite(b.sLo) && isfinite(b.sHi) && isfinite(b.wLo) && isfinite(b.wHi) &&
                        isfinite(cut) && b.wLo >= 0.f;
    b.valid = __all_sync(0xffffffffu, !(live && fc.force)) && enabled && finite && __any_sync(0xffffffffu, live);
    return b;
}

__device__ __forceinline__ bool eventCutForBox(float ls, float d, float nl2, const SkipBox& b) {
    const bool up = d >= 0.f;
    const float s = (up == (ls >= 0.f)) ? b.sLo : b.sHi;
    const float w = up ? b.wLo : b.wHi;
    const float t = __fmul_rn(d, fastEx2(__fmul_rn(ls, s)));
    const float z = __fmaf_rn(t, w, nl2);
    return z >= __fmaf_ru(fabsf(t), b.slope, b.zCut);
}

// Warp-collective: true when every event of the tile is cut for every chain of the box (each lane
// tests four events).  Padding records (nl2 = +inf) are cut.
__device__ __forceinline__ bool tileAllCut(const FilterTile* tile, const SkipBox& b, int lane) {
    const float4 ls = reinterpret_cast<const float4*>(tile->ls)[lane];
    const float4 d = reinterpret_cast<const float4*>(tile->d)[lane];
    const float4 nl = reinterpret_cast<const float4*>(tile->nl2)[lane];
    const bool cut = eventCutForBox(ls.x, d.x, nl.x, b) & eventCutForBox(ls.y, d.y, nl.y, b) &
                     eventCutForBox(ls.z, d.z, nl.z, b) & eventCutForBox(ls.w, d.w, nl.w, b);
    return __all_sync(0xffffffffu, cut);
}

// A tile of an untagged class that straddles a mass-band boundary is not sorted by separation.
__device__ __forceinline__ bool tileStraddlesBand(const PairLaunch& L, int cls, int64_t tileFirst) {
    bool straddles = false;
#pragma unroll
    for (int b = 1; b < kMassBands; ++b) {
        const int64_t s = L.bandStart[cls][b];
        straddles |= s > tileFirst && s < tileFirst + kPairTile;
    }
    return straddles;
}

template <bool TAGGED>
__device__ __forceinline__ void pairChunk(const PairLaunch& L, int cls, int64_t first, int count,
                                          int pointBase, FilterTile* tiles, uint64_t* bars,
                                          uint32_t* counters, PairQueue* queue) {
    const int tid = threadIdx.x;
    const int point = pointBase + tid;
    const bool live = point < L.numPoints;
    const bool warpLive = __any_sync(0xffffffffu, live);
    FilterChain fc;
    if (live) fc = L.filterChains[point];
    else {
        // no chain here: A = B (hi == lo for every event) and a negative bound of the separation test --
        // nothing this lane computes is ever "undecided", nothing is read from its counters
        fc.scl2 = 0.f; fc.w2 = 1.f; fc.a0 = 1.f; fc.aT = 0.f; fc.twoK = 2.f; fc.force = 0u;
        fc.thr[0] = fc.thr[1] = 100.f; fc.thrEps[0] = fc.thrEps[1] = -1.f;
    }
    const float thr = (cls >> 1) ? fc.thr[1] : fc.thr[0];
    const float thrEps = (cls >> 1) ? fc.thrEps[1] : fc.thrEps[0];
    constexpr int rows = TAGGED ? kPairCutRow : kPairCounterRows + 1;      // the cut row is cleared too, never read
    for (int w = tid; w < rows * (kPairThreads / 2); w += kPairThreads) counters[w] = 0;
    const unsigned countersAddr = smemAddr(counters);
    const int64_t classFirst = L.classBase[cls] + first;          // a multiple of kPairTile
    if (tid == 0) {
        queue->done[0] = queue->done[1] = 0;
        queue->unsure = 0;
        queue->skipped = 0;
        queue->cls = cls;
        queue->chunkEvents = L.events + classFirst;
        queue->chains = L.chains + pointBase;
        queue->countersAddr = countersAddr;
    }
    if (tid < kPairWarps) queue->count[tid] = 0;
    // chains c and c+128 share a word: the 32 lanes of a warp always address 32
    // consecutive words, i.e. 32 different banks, whatever rows they hit
    const unsigned mineWord = countersAddr + (unsigned)(tid & (kPairThreads / 2 - 1)) * 4u;
    PairRows nearRows;
    nearRows.mul = kPairRowBytes;
    nearRows.adj = mineWord - kFloorMagicBits * kPairRowBytes;
    nearRows.farMul = 0u - kPairRowBytes;
    nearRows.farAdj = mineWord + kPairFarRow0 * kPairRowBytes + kFloorMagicBits * kPairRowBytes;
    const unsigned mineAdd = (tid >= kPairThreads / 2) ? 65536u : 1u;
    // Range of the separation cut over the chains of the CTA, widened by the
    // error bound of the FP32 comparison: a tile whose separations all lie below
    // sepLow (above sepHigh) is near (far) for every chain, decided.
    float sepLow = 0.f, sepHigh = 0.f;
    if (!TAGGED) {
        const float inf = __int_as_float(0x7f800000);
        const bool usable = !(isnan(thr) || isnan(thrEps));
        float lo = live ? (usable ? __fsub_rd(thr, thrEps) : -inf) : inf;
        float hi = live ? (usable ? __fadd_ru(thr, thrEps) : inf) : -inf;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        float* red = reinterpret_cast<float*>(&queue->entry[0][0]);   // the queues are not in use yet
        if ((tid & 31) == 0) {
            red[(tid >> 5) * 2] = lo;
            red[(tid >> 5) * 2 + 1] = hi;
        }
        __syncthreads();
        sepLow = red[0];
        sepHigh = red[1];
#pragma unroll
        for (int w = 1; w < kPairThreads / 32; ++w) {
            sepLow = fminf(sepLow, red[2 * w]);
            sepHigh = fmaxf(sepHigh, red[2 * w + 1]);
        }
    }
    __syncthreads();

    const FilterTile* src = L.filterTiles + classFirst / kPairTile;
    const int numTiles = count / kPairTile;
    // The tile skip: tested on the tiles that hold events of the candidate bands (the tiles before
    // them are below the cut for any chain near the bulk of the sample, and pay nothing).
    const SkipBox box = warpSkipBox(fc, live, L.skipTiles != 0);
    const int64_t candidate = L.bandStart[cls][kFirstCandidateBand] - first;    // events into the chunk
    const int firstCandidateTile = candidate <= 0 ? 0 : (int)min((int64_t)numTiles, candidate / kPairTile);
    const unsigned livePairsPerTile = (unsigned)__popc(__ballot_sync(0xffffffffu, live)) * kPairTile;
    // Two tile buffers.  There is no CTA-wide barrier per tile: a warp that has
    // finished a tile says so with an atomic increment of done[buffer], and the
    // warp that makes the count complete refills the buffer with the tile after
    // next (TMA bulk copy, completion on the buffer's mbarrier).  Warps drift
    // apart by up to one tile instead of meeting at every tile end.
    if (tid == 0) {
        for (int b = 0; b < 2 && b < numTiles; ++b) {
            mbarExpectTx(&bars[b], (uint32_t)sizeof(FilterTile));
            tmaLoad1D(&tiles[b], src + b, (uint32_t)sizeof(FilterTile), &bars[b]);
        }
    }
    for (int t = 0; t < numTiles; ++t) {
        const int buf = t & 1;
        mbarWait(&bars[buf], (uint32_t)(t >> 1) & 1u);
        const FilterTile* tile = &tiles[buf];
        // Untagged classes: inside a mass band the events are sorted by separation, so most tiles
        // lie on one side of the cut for every chain of the CTA and the per-pair separation test
        // (and the load of the separations) is skipped there.  A tile across a band boundary is
        // not sorted: it tests every pair.
        int mode = 0;                             // 0: test every pair, 1: all near, 2: all far
        if (TAGGED) mode = 1;
        else if (tileStraddlesBand(L, cls, first + (int64_t)t * kPairTile)) mode = 0;
        else if (tile->sep[kPairTile - 1] < sepLow) mode = 1;
        else if (tile->sep[0] > sepHigh) mode = 2;
        // a warp without a live chain (ensembles that do not fill the 256-chain tile) only
        // keeps the buffer protocol going; a warp for whose whole box every event of the tile
        // is cut has nothing to count in it
        bool skip = false;
        if (box.valid && t >= firstCandidateTile) {
            skip = tileAllCut(tile, box, tid & 31);
            if (skip && L.stats && (tid & 31) == 0) atomicAdd(&queue->skipped, livePairsPerTile);
        }
        if (warpLive && !skip) {
            PairRows rows = nearRows;             // (by value: a pointer to one of two structs puts both on the stack)
            if (mode == 2) {
                rows.mul = nearRows.farMul;
                rows.adj = nearRows.farAdj;
            }
            if (mode == 0) tileLoop<false>(tile, fc, thr, thrEps, rows, mineAdd, fc.force, queue, t * kPairTile);
            else tileLoop<true>(tile, fc, thr, thrEps, rows, mineAdd, fc.force, queue, t * kPairTile);
        }
        // end of tile for this warp: release the buffer
        __syncwarp();
        if ((tid & 31) == 0) {
            __threadfence_block();
            const unsigned before = atomicAdd(&queue->done[buf], 1u);
            if (before == kPairThreads / 32 - 1) {            // the last warp of the CTA to finish tile t
                __threadfence_block();
                queue->done[buf] = 0;
                if (t + 2 < numTiles) {
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    mbarExpectTx(&bars[buf], (uint32_t)sizeof(FilterTile));
                    tmaLoad1D(&tiles[buf], src + (t + 2), (uint32_t)sizeof(FilterTile), &bars[buf]);
                }
            }
        }
        // the warp's queue of undecided pairs: worked off once enough lanes would be busy, and at the
        // end of the chunk (the count is the same for the whole warp after the barrier above)
        const unsigned queued = queue->count[tid >> 5];
        if (queued >= (unsigned)kPairDrainAt || (queued && t + 1 == numTiles)) drainWarpQueue(queue);
    }
    if (live) {
        const int slotBase = fakeClassSlotBase(cls);
        const int word = tid & (kPairThreads / 2 - 1), shift = (tid >= kPairThreads / 2) ? 16 : 0;
        constexpr int bins = TAGGED ? kFilterCutRow : 2 * kFilterCutRow;
        for (int b = 0; b < bins; ++b) {
            const uint32_t v = (counters[pairRowOfBin(b) * (kPairThreads / 2) + word] >> shift) & 0xffffu;
            if (v) atomicAdd(&L.counts[countIndex(slotBase + b, point, L.blockPoints)], v);
        }
    }
    if (L.stats) {
        __syncthreads();
        if (tid == 0 && queue->unsure) atomicAdd(&L.stats[0], (unsigned long long)queue->unsure);
        if (tid == 0 && queue->skipped) atomicAdd(&L.stats[1], (unsigned long long)queue->skipped);
    }
}

// grid.x = (#chunks over all classes) * (#point tiles); consecutive CTAs take
// the point tiles of the same chunk, so a chunk is fetched from HBM once and
// re-read from L2 by the other tiles.
__global__ void __launch_bounds__(kPairThreads, kPairCtasPerSm)
kFakePairs(const __grid_constant__ PairLaunch L) {
    extern __shared__ __align__(128) unsigned char smemRaw[];
    FilterTile* tiles = reinterpret_cast<FilterTile*>(smemRaw);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smemRaw + kPairSmemTiles);
    uint32_t* counters = reinterpret_cast<uint32_t*>(smemRaw + kPairSmemTiles + 64);
    PairQueue* queue = reinterpret_cast<PairQueue*>(smemRaw + kPairSmemTiles + 64 + kPairSmemCounters);

    const int pointTiles = (L.numPoints + kPairThreads - 1) / kPairThreads;
    const int chunk = blockIdx.x / pointTiles;
    const int pointBase = (blockIdx.x - chunk * pointTiles) * kPairThreads;
    int cls = 0;
    while (cls + 1 < kFakeClasses && chunk >= L.chunkBase[cls + 1]) ++cls;
    const int64_t first = (int64_t)(chunk - L.chunkBase[cls]) * L.chunkEvents;
    const int count = (int)min((int64_t)L.chunkEvents, L.classCount[cls] - first);

    if (threadIdx.x == 0) {
        mbarInit(&bars[0], 1);
        mbarInit(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (cls & 1) pairChunk<true>(L, cls, first, count, pointBase, tiles, bars, counters, queue);
    else pairChunk<false>(L, cls, first, count, pointBase, tiles, bars, counters, queue);
}

// ---------------------------------------------------------------------------
// The streaming kernel: FEW chains (<= kStreamMaxChains) over many events.
//
// kFakePairs maps one chain to one thread and reuses every event tile for 256
// chains: with a handful of chains (the reference's own use: ONE chain) 255 of
// its 256 threads idle.  Here the roles are swapped: a warp takes one tile of
// 128 events (four per lane, the tile's 2 KB read with four coalesced 16-byte
// loads per lane), every lane evaluates its four events for each of the E chains
// (parameters in shared memory) with the same FP32 interval filter and the same
// FP64 fallback, and counts into a per-CTA shared-memory table that is flushed
// to the global count table at the end.  Each event is read ONCE: 16 bytes per
// event per evaluation, HBM-bound for E <= ~4 (SURVEY.md 8d "streaming regime").
// The counts are the same integers kFakePairs produces.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void fakePairGeneric(const smcmc_event& e, const double* __restrict__ p, int point,
                                                uint32_t* counts, int blockPoints);
constexpr int kStreamMaxChains = 16;
constexpr int kStreamThreads = 256;
constexpr int kStreamRows = 300;             // slots of the four weight classes

template <bool TAGGED>
__device__ __forceinline__ void streamCount(const FilterDecision& dec, int cls, int chain, int64_t event,
                                            const PairLaunch& L, const FakeChainParams* cps, uint32_t* table) {
    int row;
    if (dec.sure) {
        if (!dec.counted) return;
        row = (int)(dec.bits - kFloorMagicBits);
        if (!TAGGED && dec.far) row += 50;
    } else {
        row = exactDecide(L.events[event], cps[chain], cls);             // FP64, the reference's arithmetic
        if (row < 0) return;
    }
    atomicAdd(&table[chain * kStreamRows + fakeClassSlotBase(cls) + row], 1u);
}

// a lane's four events of one tile (four coalesced 16-byte loads; the separation only for the untagged classes)
struct StreamRegs {
    float4 ls, d, nl, sp;
};
template <bool TAGGED>
__device__ __forceinline__ StreamRegs streamLoad(const PairLaunch& L, int64_t tileIndex, int lane) {
    const FilterTile& tile = L.filterTiles[tileIndex];
    StreamRegs r;
    r.ls = __ldcs(reinterpret_cast<const float4*>(tile.ls) + lane);      // read once: streaming loads
    r.d = __ldcs(reinterpret_cast<const float4*>(tile.d) + lane);
    r.nl = __ldcs(reinterpret_cast<const float4*>(tile.nl2) + lane);
    r.sp = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!TAGGED) r.sp = __ldcs(reinterpret_cast<const float4*>(tile.sep) + lane);
    return r;
}

template <bool TAGGED>
__device__ __forceinline__ void streamTile(const PairLaunch& L, int cls, int64_t tileIndex, int lane, const StreamRegs& regs,
                                           const FilterChain* fcs, const FakeChainParams* cps, uint32_t* table) {
    const float4 ls = regs.ls, d = regs.d, nl = regs.nl, sp = regs.sp;
    const int64_t event0 = tileIndex * kPairTile + 4 * lane;
    for (int c = 0; c < L.numPoints; ++c) {
        const FilterChain fc = fcs[c];
        const float thr = fc.thr[cls >> 1], thrEps = fc.thrEps[cls >> 1];
        const FilterPair a = filterCore2<TAGGED>(make_float2(ls.x, ls.y), make_float2(d.x, d.y), make_float2(nl.x, nl.y),
                                                 make_float2(sp.x, sp.y), fc, thr);
        const FilterPair b = filterCore2<TAGGED>(make_float2(ls.z, ls.w), make_float2(d.z, d.w), make_float2(nl.z, nl.w),
                                                 make_float2(sp.z, sp.w), fc, thr);
        streamCount<TAGGED>(filterDecide<TAGGED>(a.lo.x, a.hi.x, a.ds.x, thrEps), cls, c, event0 + 0, L, cps, table);
        streamCount<TAGGED>(filterDecide<TAGGED>(a.lo.y, a.hi.y, a.ds.y, thrEps), cls, c, event0 + 1, L, cps, table);
        streamCount<TAGGED>(filterDecide<TAGGED>(b.lo.x, b.hi.x, b.ds.x, thrEps), cls, c, event0 + 2, L, cps, table);
        streamCount<TAGGED>(filterDecide<TAGGED>(b.lo.y, b.hi.y, b.ds.y, thrEps), cls, c, event0 + 3, L, cps, table);
    }
}

// PREFETCH: the loads of a warp's next tile are in flight while the current one is evaluated
// (80 registers, three CTAs per SM) or not (54 registers, four CTAs per SM)
template <bool PREFETCH>
__global__ void __launch_bounds__(kStreamThreads, PREFETCH ? 3 : 4)
kFakeStream(const __grid_constant__ PairLaunch L) {
    __shared__ uint32_t table[kStreamMaxChains * kStreamRows];
    __shared__ FilterChain fcs[kStreamMaxChains];
    __shared__ FakeChainParams cps[kStreamMaxChains];
    for (int k = threadIdx.x; k < L.numPoints * kStreamRows; k += kStreamThreads) table[k] = 0u;
    if (threadIdx.x < L.numPoints) {
        fcs[threadIdx.x] = L.filterChains[threadIdx.x];
        cps[threadIdx.x] = L.chains[threadIdx.x];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * (kStreamThreads / 32) + (threadIdx.x >> 5);
    const int64_t warps = (int64_t)gridDim.x * (kStreamThreads / 32);
    for (int cls = 0; cls < kFakeClasses; ++cls) {
        const int64_t firstTile = L.classBase[cls] / kPairTile;
        const int64_t tiles = L.classCount[cls] / kPairTile;             // padded to whole tiles
        if (!PREFETCH) {
            for (int64_t t = warp; t < tiles; t += warps) {
                if (cls & 1) streamTile<true>(L, cls, firstTile + t, lane, streamLoad<true>(L, firstTile + t, lane), fcs, cps, table);
                else streamTile<false>(L, cls, firstTile + t, lane, streamLoad<false>(L, firstTile + t, lane), fcs, cps, table);
            }
        } else if (cls & 1) {
            StreamRegs nxt;
            if (warp < tiles) nxt = streamLoad<true>(L, firstTile + warp, lane);
            for (int64_t t = warp; t < tiles; t += warps) {
                const StreamRegs cur = nxt;
                if (t + warps < tiles) nxt = streamLoad<true>(L, firstTile + t + warps, lane);
                streamTile<true>(L, cls, firstTile + t, lane, cur, fcs, cps, table);
            }
        } else {
            StreamRegs nxt;
            if (warp < tiles) nxt = streamLoad<false>(L, firstTile + warp, lane);
            for (int64_t t = warp; t < tiles; t += warps) {
                const StreamRegs cur = nxt;
                if (t + warps < tiles) nxt = streamLoad<false>(L, firstTile + t + warps, lane);
                streamTile<false>(L, cls, firstTile + t, lane, cur, fcs, cps, table);
            }
        }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < L.numPoints * kStreamRows; k += kStreamThreads) {
        const uint32_t v = table[k];
        if (v) {
            const int c = k / kStreamRows, slot = k - c * kStreamRows;
            atomicAdd(&L.counts[countIndex(slot, c, L.blockPoints)], v);
        }
    }
}

// Test kernel: run the filter AND the FP64 arithmetic on every pair and count
// the pairs where a filter decision differs from the FP64 decision (must be
// zero).  stats[0] = pairs, [1] = unsure, [2] = mismatches.
__global__ void kFakeVerifyFilter(const PairLaunch L, unsigned long long* stats) {
    const int point = blockIdx.y * blockDim.x + threadIdx.x;
    if (point >= L.numPoints) return;
    const FakeChainParams cp = L.chains[point];
    const FilterChain fc = L.filterChains[point];
    unsigned long long pairs = 0, unsure = 0, bad = 0;
    for (int cls = 0; cls < kFakeClasses; ++cls) {
        const float thr = (cls >> 1) ? fc.thr[1] : fc.thr[0];
        const float thrEps = (cls >> 1) ? fc.thrEps[1] : fc.thrEps[0];
        for (int64_t i = blockIdx.x; i < L.classReal[cls]; i += gridDim.x) {
            const int64_t idx = L.classBase[cls] + i;
            const FilterTile& tile = L.filterTiles[idx / kPairTile];
            const int k = (int)(idx % kPairTile);
            const float2 ls = make_float2(tile.ls[k], tile.ls[k]), d = make_float2(tile.d[k], tile.d[k]);
            const float2 nl = make_float2(tile.nl2[k], tile.nl2[k]), sp = make_float2(tile.sep[k], tile.sep[k]);
            FilterDecision r;
            if (cls & 1) {
                const FilterPair fp = filterCore2<true>(ls, d, nl, sp, fc, thr);
                r = filterDecide<true>(fp.lo.y, fp.hi.y, fp.ds.y, thrEps);
            } else {
                const FilterPair fp = filterCore2<false>(ls, d, nl, sp, fc, thr);
                r = filterDecide<false>(fp.lo.y, fp.hi.y, fp.ds.y, thrEps);
            }
            const int f = r.counted ? (int)(r.bits - kFloorMagicBits) + (r.far ? kFilterCutRow : 0) : -1;
            const int x = exactDecide(L.events[idx], cp, cls);
            ++pairs;
            if (!r.sure) ++unsure;
            else if (f != x) ++bad;
        }
    }
    atomicAdd(&stats[0], pairs);
    atomicAdd(&stats[1], unsure);
    atomicAdd(&stats[2], bad);
}

// Test kernel for the tile skip: for each warp of 32 consecutive points (blockIdx.y * 4 + warp) and
// each tile of the candidate bands, the pair kernel's skip rule (warpSkipBox, tileAllCut), and for
// every pair of every skipped tile the FP64 decision, which must be "cut".  stats[0] = tiles
// tested, [1] = tiles skipped, [2] = pairs of skipped tiles that exactDecide counts (must be zero).
__global__ void kFakeSkipCheck(const __grid_constant__ PairLaunch L, unsigned long long* stats) {
    const int lane = threadIdx.x & 31;
    const int point = (blockIdx.y * (blockDim.x / 32) + (threadIdx.x >> 5)) * 32 + lane;
    if (__all_sync(0xffffffffu, point >= L.numPoints)) return;
    const bool live = point < L.numPoints;
    FilterChain fc = {};
    FakeChainParams cp = {};
    if (live) {
        fc = L.filterChains[point];
        cp = L.chains[point];
    }
    const SkipBox box = warpSkipBox(fc, live, L.skipTiles != 0);
    if (!box.valid) return;
    unsigned long long tested = 0, skipped = 0, bad = 0;
    for (int cls = 0; cls < kFakeClasses; ++cls) {
        const int64_t firstTile = L.bandStart[cls][kFirstCandidateBand] / kPairTile;
        const int64_t tiles = L.classCount[cls] / kPairTile;
        for (int64_t t = firstTile + blockIdx.x; t < tiles; t += gridDim.x) {
            const FilterTile* tile = L.filterTiles + L.classBase[cls] / kPairTile + t;
            ++tested;
            if (!tileAllCut(tile, box, lane)) continue;
            ++skipped;
            if (!live) continue;
            for (int k = 0; k < kPairTile; ++k)
                if (exactDecide(L.events[L.classBase[cls] + t * kPairTile + k], cp, cls) >= 0) ++bad;
        }
    }
    if (lane == 0) {
        atomicAdd(&stats[0], tested);
        atomicAdd(&stats[1], skipped);
    }
    if (bad) atomicAdd(&stats[2], bad);
}

// Straight transcription of the per-event formula for the events the fast
// path cannot take (data-typed, negative separation, non-finite fields):
// one thread per (point, event).
__device__ __forceinline__ void fakePairGeneric(const smcmc_event& e, const double* __restrict__ p, int point,
                                                uint32_t* counts, int blockPoints);

__global__ void kFakePairsGeneric(const smcmc_event* __restrict__ ev, int64_t nev,
                                  const double* __restrict__ x, int m, int dim,
                                  uint32_t* counts, int blockPoints) {
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nev * (int64_t)m) return;
    int point = (int)(idx % m);
    fakePairGeneric(ev[idx / m], x + (size_t)point * dim, point, counts, blockPoints);
}

__device__ __forceinline__ void fakePairGeneric(const smcmc_event& e, const double* __restrict__ p, int point,
                                                uint32_t* counts, int blockPoints) {
    double mass = e.Mass, sep = e.Separation;
    if (e.Type >= 0) {
        double nomLog = log(e.TrueMass);
        double nomLogSigma = __dsub_rn(log(__dadd_rn(e.TrueMass, e.TrueMassSigma)), nomLog);
        double logMass = log(mass);
        double logSigma = __ddiv_rn(__dsub_rn(logMass, nomLog), nomLogSigma);
        double scale = __ddiv_rn(p[2], 10.0);
        double width = exp(__ddiv_rn(p[3], 10.0));
        double skew = __dmul_rn(0.3, erf(__ddiv_rn(p[4], 10.0)));
        skew = exp(__dmul_rn(logSigma, skew));
        logMass = __dadd_rn(nomLog, __dmul_rn(__dsub_rn(logMass, nomLog), skew));
        logMass = __dadd_rn(nomLog, __dmul_rn(__dsub_rn(logMass, nomLog), width));
        logMass = __dadd_rn(logMass, scale);
        double sc = exp(__ddiv_rn(__dadd_rn(0.0, e.Type == 0 ? p[5] : p[6]), 10.0));
        sep = __dmul_rn(sep, sc);
        if (sep < 0.0) return;
        int bin = exactBin(logMass, 25);
        if (bin >= 50) return;
        int cls = (e.Type == 0 ? 0 : 2) + (e.MuDk > 0 ? 1 : 0);
        int row = bin;
        if (!(cls & 1) && !(sep < 100.0)) row += 50;
        atomicAdd(&counts[countIndex(fakeClassSlotBase(cls) + row, point, blockPoints)], 1u);
    } else {
        if (mass > 500.0 || mass < 0.0 || sep < 0.0) return;
        if (!(mass < 500.0)) return;                 // NaN or ==500: overflow bin
        int bin = (int)(50 * (mass - 0.0) / (500.0 - 0.0));
        int h = e.MuDk > 0 ? 2 : (sep < 100.0 ? 0 : 1);
        atomicAdd(&counts[countIndex(300 + h * 50 + bin, point, blockPoints)], 1u);
    }
}

// ---------------------------------------------------------------------------
// Counts -> bin contents -> log-likelihood (FakeLikelihood.H:51-80).
// The work is 150 x m independent (point, bin) items, each three emulated running
// sums (seqsum.h: data-dependent loops with an FP64 division per binade) and a
// log: latency-bound, so the kernel wants as many warps as the SMs hold.  Block =
// kFinishPoints points x kFinishBinWarps warps; a warp covers two bins for 16
// points (lane & 15 = point, lane >> 4 = bin parity).  4096 points: 256 CTAs x 15
// warps: 0.151 -> 0.058 ms per launch (DESIGN.md 4.2).
// ---------------------------------------------------------------------------
constexpr int kFinishWarps = 30;            // kFake2Finish: 32 points x 30 warps over the 150 bins (was 10: 9 warps per SM)
constexpr int kFinishPoints = 16;
constexpr int kFinishBinWarps = 15;

// With few points the grid's y dimension splits the 150 bins over kFinishGroups
// CTAs (one item per thread: the latency of ONE item instead of five); the terms
// go through global memory and the last CTA of a point group to arrive (ticket
// counter, reset by that CTA) adds them in bin order.
constexpr int kFinishGroups = 5;

__global__ void __launch_bounds__(32 * kFinishBinWarps)
kFakeFinish(const uint32_t* __restrict__ counts, int pointStride, int m,
            const FakeChainParams* __restrict__ chains, const double* __restrict__ data150,
            double* llhOut, double* histOut, double* termScratch, unsigned int* tickets) {
    __shared__ double term[150][kFinishPoints + 1];
    __shared__ int lastArriver;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int p = lane & (kFinishPoints - 1);
    const int sub = lane / kFinishPoints;                   // 0 or 1
    const int point = blockIdx.x * kFinishPoints + p;
    const bool live = point < m;
    const int groups = gridDim.y;
    const int binsPerGroup = 150 / groups;
    const int binBase = blockIdx.y * binsPerGroup;
    double w[4] = {0, 0, 0, 0};
    if (live) {
        for (int k = 0; k < 4; ++k) w[k] = chains[point].weight[k];
    }
    for (int hb = binBase + 2 * warp + sub; hb < binBase + binsPerGroup; hb += 2 * kFinishBinWarps) {
        const int h = hb / 50, b = hb - h * 50;
        double v = 0.0;
        if (live) {
            uint32_t nSig, nBkg, nDat;
            double wSig, wBkg;
            if (h < 2) {
                nSig = counts[(size_t)(0 + h * 50 + b) * pointStride + point];
                nBkg = counts[(size_t)(150 + h * 50 + b) * pointStride + point];
                wSig = w[0];
                wBkg = w[2];
            } else {
                nSig = counts[(size_t)(100 + b) * pointStride + point];
                nBkg = counts[(size_t)(250 + b) * pointStride + point];
                wSig = w[1];
                wBkg = w[3];
            }
            nDat = counts[(size_t)(300 + hb) * pointStride + point];
            // TH1::Fill in event order: the signal block, then the background
            // block (Simulated::MakeSample, example/Simulated.H:17-29).
            double mc = smcmc_seq_add(0.0, wSig, nSig);
            mc = smcmc_seq_add(mc, wBkg, nBkg);
            mc = smcmc_seq_add(mc, 1.0, nDat);
            if (histOut) histOut[(size_t)point * 150 + hb] = mc;
            const double d = data150[hb];
            if (mc < 0.001) mc = 0.001;                                 // :56
            v = __dsub_rn(d, mc);                                       // :57
            if (d > 0.0) v = __dadd_rn(v, __dmul_rn(d, log(__ddiv_rn(mc, d))));   // :58
        }
        if (groups == 1) term[hb][p] = v;
        else if (live) termScratch[(size_t)point * 150 + hb] = v;
    }
    if (groups > 1) {
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned int ticket = atomicAdd(tickets + blockIdx.x, 1u);
            lastArriver = ticket == (unsigned int)(groups - 1);
            if (lastArriver) tickets[blockIdx.x] = 0;                   // ready for the next evaluation
        }
        __syncthreads();
        if (!lastArriver) return;
        __threadfence();
        // the terms come back through shared memory, every thread fetching a few in parallel: the
        // ordered sum below then waits for LDS, not for 150 round trips to L2 one after the other
        for (int k = threadIdx.x; k < 150 * kFinishPoints; k += blockDim.x) {
            const int hb = k / kFinishPoints, pp = k - hb * kFinishPoints;
            const int pt = blockIdx.x * kFinishPoints + pp;
            if (pt < m) term[hb][pp] = __ldcg(termScratch + (size_t)pt * 150 + hb);
        }
        __syncthreads();
        if (warp == 0 && sub == 0 && live && llhOut) {
            double s = 0.0;
#pragma unroll 6
            for (int hb = 0; hb < 150; ++hb) s = __dadd_rn(s, term[hb][p]);
            llhOut[point] = s;
        }
        return;
    }
    __syncthreads();
    if (warp == 0 && sub == 0 && live && llhOut) {
        double s = 0.0;                                                 // :51,59 in bin order
#pragma unroll 6
        for (int hb = 0; hb < 150; ++hb) s = __dadd_rn(s, term[hb][p]);
        llhOut[point] = s;
    }
}

// ---------------------------------------------------------------------------
// example2/FakeLikelihood.H: counts -> the six signal / background histograms ->
// their integrals -> renormalised expectation (:266-288) -> log-likelihood and
// penalty terms (:58-118).  Block = 32 points (lane = point) x kFinishWarps warps
// striding the 150 bins; dynamic shared memory 2 x 150 x 33 doubles.
// Event order as in kFakeFinish: background events, then data-typed ones (which
// IsSignal() sends to the background histograms with weight 1).
// ---------------------------------------------------------------------------
constexpr size_t kFinish2SmemBytes = (size_t)2 * 150 * 33 * sizeof(double);

__global__ void __launch_bounds__(32 * kFinishWarps)
kFake2Finish(const uint32_t* __restrict__ counts, int pointStride, int m,
             const FakeChainParams* __restrict__ chains, const double* __restrict__ data150,
             const double* __restrict__ x, int dim, double* llhOut, double* histOut) {
    extern __shared__ double fin2[];
    double (*sig)[33] = reinterpret_cast<double (*)[33]>(fin2);              // later: the bin terms
    double (*bkg)[33] = reinterpret_cast<double (*)[33]>(fin2 + 150 * 33);
    __shared__ double norm[2][32];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int point = blockIdx.x * 32 + lane;
    const bool live = point < m;
    double w[4] = {0, 0, 0, 0};
    if (live) {
        for (int k = 0; k < 4; ++k) w[k] = chains[point].weight[k];
    }
    for (int hb = warp; hb < 150; hb += kFinishWarps) {
        const int h = hb / 50, b = hb - h * 50;
        double s = 0.0, g = 0.0;
        if (live) {
            uint32_t nSig, nBkg;
            double wSig, wBkg;
            if (h < 2) {
                nSig = counts[(size_t)(0 + h * 50 + b) * pointStride + point];
                nBkg = counts[(size_t)(150 + h * 50 + b) * pointStride + point];
                wSig = w[0];
                wBkg = w[2];
            } else {
                nSig = counts[(size_t)(100 + b) * pointStride + point];
                nBkg = counts[(size_t)(250 + b) * pointStride + point];
                wSig = w[1];
                wBkg = w[3];
            }
            const uint32_t nDat = counts[(size_t)(300 + hb) * pointStride + point];
            s = smcmc_seq_add(0.0, wSig, nSig);                          // Simulated*Signal      :244-262
            g = smcmc_seq_add(0.0, wBkg, nBkg);                          // Simulated*Background
            g = smcmc_seq_add(g, 1.0, nDat);
        }
        sig[hb][lane] = s;
        bkg[hb][lane] = g;
    }
    __syncthreads();
    if (warp == 0 && live) {
        // TH1::Integral: bins 1..50 in order; DecayTag, Close, Separated (:266-277)
        const double* p = x + (size_t)point * dim;
        double tot[2];
        for (int k = 0; k < 2; ++k) {
            double (*hst)[33] = k ? bkg : sig;
            double part[3];
            for (int h = 0; h < 3; ++h) {
                double t = 0.0;
                for (int b = 0; b < 50; ++b) t = __dadd_rn(t, hst[h * 50 + b][lane]);
                part[h] = t;
            }
            double t = part[2];
            t = __dadd_rn(t, part[0]);
            t = __dadd_rn(t, part[1]);
            tot[k] = __ddiv_rn(p[k], t);                                 // :269-270, :276-277
        }
        norm[0][lane] = tot[0];
        norm[1][lane] = tot[1];
    }
    __syncthreads();
    for (int hb = warp; hb < 150; hb += kFinishWarps) {
        double v = 0.0;
        if (live) {
            // TH1::Add on the reset histogram: (0 + sW s) + bW b              :280-287
            double mc = __dadd_rn(0.0, __dmul_rn(norm[0][lane], sig[hb][lane]));
            mc = __dadd_rn(mc, __dmul_rn(norm[1][lane], bkg[hb][lane]));
            if (histOut) histOut[(size_t)point * 150 + hb] = mc;
            const double d = data150[hb];
            if (mc < 0.001) mc = 0.001;                                  // :66
            v = __dsub_rn(d, mc);
            if (d > 0.0) v = __dadd_rn(v, __dmul_rn(d, log(__ddiv_rn(mc, d))));
        }
        sig[hb][lane] = v;
    }
    __syncthreads();
    if (warp == 0 && live && llhOut) {
        const double* p = x + (size_t)point * dim;
        double L = 0.0;
        for (int hb = 0; hb < 150; ++hb) L = __dadd_rn(L, sig[hb][lane]);
        if (p[0] < 0.0) L = __dsub_rn(L, __dadd_rn(10.0, fabs(L)));       // :95-96
        if (p[1] < 0.0) L = __dsub_rn(L, __dadd_rn(10.0, fabs(L)));       // :99-100
        double v = __ddiv_rn(p[6], 5.0);                                   // :104-105
        L = __dsub_rn(L, __dmul_rn(__dmul_rn(0.5, v), v));
        v = __ddiv_rn(p[7], 1.0);                                          // :109-110
        L = __dsub_rn(L, __dmul_rn(__dmul_rn(0.5, v), v));
        v = __ddiv_rn(p[8], 1.0);                                          // :114-115
        L = __dsub_rn(L, __dmul_rn(__dmul_rn(0.5, v), v));
        llhOut[point] = L;
    }
}

}  // namespace smcmc
