// user_events.cuh -- event functors written the way a user writes one
// (include/smcmc_device_functor.cuh, "EVENT functors"): the kernels are
// instantiated from these types in the translation unit that includes this file.
//
//   GaussEvents          the mean and width of a Gaussian sample, x = (mu, sigma)
//   PaddedGaussEvents<E> the same with event records of awkward sizes
//   UnbinnedEvents       the unbinned mixture likelihood of SMCMC_LLH_UNBINNED
//                        (include/smcmc_b200.h) restated as a user functor over
//                        events prepared on the host
//   UnbinnedLoop         the same likelihood as a chain-local functor that loops
//                        over a device pointer to the events from one thread per
//                        point: what an event likelihood looks like without the
//                        event kind, kept as a contrast for the benchmark
#pragma once
#include <cmath>
#include <cstdint>

#include "smcmc_device_functor.cuh"

// log with + - * / and frexp (exact) only: the host and the device round it alike,
// so the host restatement of GaussEvents is bit-identical to the device.
__host__ __device__ inline double PortableLog(double x) {
    if (x != x || x < 0.0) return (x - x) / (x - x);        // NaN
    if (x == 0.0) return -1.0 / x;                         // -inf
    if (x - x != 0.0) return x;                            // +inf
    int e;
    double m = frexp(x, &e);                               // x = m 2^e, m in [1/2, 1)
    if (m < 0.70710678118654752440) {
        m = m * 2.0;
        e = e - 1;
    }
    const double s = (m - 1.0) / (m + 1.0), s2 = s * s;    // |s| <= 0.172: log m = 2 atanh s
    double p = 1.0 / 25.0;
    for (int k = 11; k >= 0; --k) p = p * s2 + 1.0 / (2 * k + 1);
    const double ln2Hi = 6.93147180369123816490e-01, ln2Lo = 1.90821492927058770002e-10;
    return (double)e * ln2Hi + ((double)e * ln2Lo + 2.0 * s * p);
}

struct GaussEvents {
    struct Event {
        double v;
    };
    struct Chain {
        double mu, k, sigma;
    };
    __host__ __device__ Chain Prepare(const double* x, int) const {
        Chain c;
        c.mu = x[0];
        c.sigma = x[1];
        c.k = -0.5 / (x[1] * x[1]);
        return c;
    }
    __host__ __device__ double Term(const Chain& c, const Event& ev) const {
        const double d = ev.v - c.mu;
        return c.k * (d * d);
    }
    __host__ __device__ double Finish(const Chain& c, double sum, int64_t n) const {
        return sum - (double)n * PortableLog(c.sigma);
    }
};

// 12 bytes, 4-byte aligned
struct Event12 {
    float v;
    float w;
    int32_t k;
    __host__ __device__ double Value() const { return (double)v; }
    __host__ __device__ double Extra() const { return (double)w * (double)k; }
};
// 128 bytes, the largest event record
struct Event128 {
    double v[16];
    __host__ __device__ double Value() const { return v[0]; }
    __host__ __device__ double Extra() const { return v[15] - v[7]; }
};

template <class E>
struct PaddedGaussEvents {
    typedef E Event;
    typedef GaussEvents::Chain Chain;
    __host__ __device__ Chain Prepare(const double* x, int n) const { return GaussEvents().Prepare(x, n); }
    __host__ __device__ double Term(const Chain& c, const Event& ev) const {
        const double d = ev.Value() - c.mu;
        return c.k * (d * d) + ev.Extra();
    }
    __host__ __device__ double Finish(const Chain& c, double sum, int64_t n) const {
        return GaussEvents().Finish(c, sum, n);
    }
};

// SMCMC_LLH_UNBINNED (csrc/unbinned_likelihood.cuh: kUnbinnedPrepareChains,
// kUnbinnedPairs) with the per-event corrections prepared on the host:
//   nomLog = log M0, dLog = log m - nomLog, logSigma = dLog / (log(M0 + S0) - nomLog),
//   tag = MuDk > 0.
struct UnbinnedEvents {
    struct Event {
        double logSigma;
        double dLog;
        double nomLog;
        int32_t tag;
        int32_t pad;
    };
    struct Chain {
        double skewc, width, scale;
        double la0, la1, lb0, lb1;     // log weight + log normalisation: untagged, tagged
    };
    // host values, set by Init()
    double tanFakes, tanEff, pi, mu, invSig, invTau, ca, cb;

    void Init() {
        pi = M_PI;
        tanFakes = std::tan(M_PI * (0.05 - 0.5));
        tanEff = std::tan(M_PI * (0.5 - 0.5));
        mu = std::log(135.0);
        invSig = 1.0 / std::log(1.3);
        invTau = 1.0 / 500.0;
        ca = -std::log(std::log(1.3) * std::sqrt(2.0 * M_PI));
        cb = -std::log(500.0);
    }
    __host__ __device__ Chain Prepare(const double* p, int) const {
        Chain u;
        u.scale = p[2] / 10.0;
        u.width = exp(p[3] / 10.0);
        u.skewc = 0.3 * erf(p[4] / 10.0);
        const double fakes = atan(tanFakes + p[7]) / pi + 0.5;
        const double eff = atan(tanEff + p[8]) / pi + 0.5;
        const double wSig = exp(p[0] / 10.0), wBkg = exp(p[1] / 10.0);
        u.la0 = log(wSig * ((1.0 - fakes) / (1.0 - 0.05))) + ca;
        u.la1 = log(wSig * (fakes / 0.05)) + ca;
        u.lb0 = log(wBkg * ((1.0 - eff) / (1.0 - 0.5))) + cb;
        u.lb1 = log(wBkg * (eff / 0.5)) + cb;
        return u;
    }
    __host__ __device__ double Term(const Chain& c, const Event& ev) const {
        const double la = ev.tag ? c.la1 : c.la0, lb = ev.tag ? c.lb1 : c.lb0;
        const double skew = exp(ev.logSigma * c.skewc);
        double lm = ev.nomLog + ev.dLog * skew;
        lm = ev.nomLog + (lm - ev.nomLog) * c.width;
        lm = lm + c.scale;
        const double z = (lm - mu) * invSig;
        const double a = la - 0.5 * z * z - lm;
        const double b = lb - exp(lm) * invTau;
        const double hi = fmax(a, b), lo = fmin(a, b);
        return hi + log1p(exp(lo - hi));      // NaN for an event with a non-positive mass
    }
};

struct UnbinnedLoop {
    UnbinnedEvents u;
    const UnbinnedEvents::Event* events;     // device pointer
    int64_t n;
    __host__ __device__ double operator()(const double* x, int dim) const {
        const UnbinnedEvents::Chain c = u.Prepare(x, dim);
        double s = 0.0;
        for (int64_t i = 0; i < n; ++i) s += u.Term(c, events[i]);
        return s;
    }
};
