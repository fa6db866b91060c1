// user_weighted.cuh -- WEIGHTED binned event functors written the way a user
// writes one (include/smcmc_device_functor.cuh, "WEIGHTED binned event functors"):
// kWeightedPairs and kWeightedFinish are instantiated from these types in the
// translation unit that includes this file.
//
//   GaussWeighted  a template fit with per-event, per-point weights: a flat
//                  template reweighted to N(x0, x1), histogrammed in GaussBinned's
//                  40 bins and compared with a data histogram held in the functor
//   FakeWeighted   example/FakeLikelihood.H's FillFake and EvalFake: the weight
//                  of every event summed into the three 50-bin histograms, then
//                  the clamped Poisson sum against the data
//   RawWeighted    the bin and the weight are carried by the event
#pragma once
#include <cmath>
#include <cstdint>

#include "user_binned.cuh"

// exp with + - * / floor and ldexp (exact) only: the host and the device round it
// alike, so GaussWeighted's host restatement is bit-identical to the device.
__host__ __device__ inline double PortableExp(double x) {
    if (x != x) return x;
    if (x > 709.0) return x * 1e308;                       // +inf
    if (x < -700.0) return 0.0;                            // keeps ldexp away from subnormals
    const double k = floor(x * 1.44269504088896338700 + 0.5);
    const double ln2Hi = 6.93147180369123816490e-01, ln2Lo = 1.90821492927058770002e-10;
    const double r = (x - k * ln2Hi) - k * ln2Lo;          // |r| <= 0.35
    double p = 1.0;
#pragma unroll
    for (int i = 18; i >= 1; --i) p = 1.0 + r * p * (1.0 / (double)i);   // constant reciprocals: no division
    return ldexp(p, (int)k);
}

struct GaussWeighted {
    struct Event {
        double u;                 // a template value, uniform over the 40 bins' range
    };
    struct Chain {
        double mu, invSigma, norm;
    };
    static constexpr int kBins = 40;
    static constexpr double kLo = -7.0, kWidth = 0.5, kRange = 20.0;   // bins over [-7, 13)
    double data[kBins];           // the data histogram
    double dataTotal;             // its sum

    __host__ __device__ Chain Prepare(const double* x, int) const {
        Chain c;
        c.mu = x[0];
        c.invSigma = 1.0 / x[1];
        c.norm = kRange * 0.39894228040143267794 / x[1];   // flat density 1/kRange -> N(mu, sigma)
        return c;
    }
    __host__ __device__ int Bin(const Chain&, const Event& ev) const {
        const double u = (ev.u - kLo) / kWidth;
        if (!(u >= 0.0 && u < (double)kBins)) return -1;
        return (int)floor(u);
    }
    // the importance weight N(u; mu, sigma) / U(u; -7, 13)
    __host__ __device__ double Weight(const Chain& c, const Event& ev) const {
        const double z = (ev.u - c.mu) * c.invSigma;
        return c.norm * PortableExp(-0.5 * z * z);
    }
    // Poisson log-likelihood (up to a constant) of the data given the reweighted
    // template scaled to the data's total, with the reference's floor on an empty bin
    __host__ __device__ double Finish(const Chain&, const smcmc_user::BinSums& sums, int64_t n) const {
        const double scale = n > 0 ? dataTotal / (double)n : 0.0;
        double s = 0.0;
        for (int b = 0; b < kBins; ++b) {
            double mu = sums[b] * scale;
            if (mu < 0.001) mu = 0.001;
            s = s + (data[b] * PortableLog(mu) - mu);
        }
        return s;
    }
};

// FillFake + EvalFake (FakeLikelihood.H:47-81, :188-216).  The bin decision is
// FakeBinned's (equal to the built-in's on every pair), mapped to the reference's
// histograms: h * 50 + bin - 1 with h = 0 Close, 1 Separated, 2 DecayTag.  The
// weight is EventWeight for the event's type and decay tag, from the per-class
// weights FakeBinned::Prepare computes in the reference's order.  A data-typed
// event (Type < 0) has weight 1 and a bin that no parameter moves, found on the
// host.
struct FakeWeighted {
    struct Event {
        double logSigma, dLog, nomLog, sep;   // as FakeBinned::Event
        int32_t cls;              // weight class 0..3, -1 for a data-typed event
        int32_t dataBin;          // a data-typed event's bin, -1 if cut
    };
    typedef FakeBinned::Chain Chain;
    static constexpr int kBins = 150;
    FakeBinned fake;              // bin edges, weight constants, data histogram

    static Event PrepareEvent(const smcmc_event& e) {
        const FakeBinned::Event f = FakeBinned::PrepareEvent(e);
        Event p;
        p.logSigma = f.logSigma;
        p.dLog = f.dLog;
        p.nomLog = f.nomLog;
        p.sep = f.sep;
        p.cls = f.cls;
        p.dataBin = -1;
        if (e.Type < 0 && !(e.Mass > 500.0) && !(e.Mass < 0.0) && !(e.Separation < 0.0)) {
            const int b = !(e.Mass < 500.0) ? 51 : 1 + int(50 * (e.Mass - 0.0) / (500.0 - 0.0));   // FindBin
            const int h = e.MuDk > 0 ? 2 : e.Separation < 100.0 ? 0 : 1;
            if (b >= 1 && b <= 50) p.dataBin = h * 50 + b - 1;
        }
        return p;
    }
    void Init(const double* data150, double exposureRatio) { fake.Init(data150, exposureRatio); }

    __host__ __device__ Chain Prepare(const double* x, int n) const { return fake.Prepare(x, n); }
    __host__ __device__ int Bin(const Chain& c, const Event& ev) const {
        if (ev.cls < 0) return ev.dataBin;
        FakeBinned::Event f;
        f.logSigma = ev.logSigma;
        f.dLog = ev.dLog;
        f.nomLog = ev.nomLog;
        f.sep = ev.sep;
        f.cls = ev.cls;
        f.pad = 0;
        const int slot = fake.Bin(c, f);
        if (slot < 0) return -1;
        return slot < 150 ? slot : slot - 150;   // background slots [150, 300) onto the same histograms
    }
    __host__ __device__ double Weight(const Chain& c, const Event& ev) const {
        return ev.cls == 0 ? c.weight[0] : ev.cls == 1 ? c.weight[1] : ev.cls == 2 ? c.weight[2]
               : ev.cls == 3 ? c.weight[3] : 1.0;   // selects, not a local-memory index
    }
    __host__ __device__ double Finish(const Chain&, const smcmc_user::BinSums& sums, int64_t) const {
        double s = 0.0;
        for (int hb = 0; hb < 150; ++hb) {
            const double d = fake.data[hb];
            double mc = sums[hb];
            if (mc < 0.001) mc = 0.001;
            double v = d - mc;
            if (d > 0.0) v = v + d * log(mc / d);
            s = s + v;
        }
        return s;
    }
};

// The bin and the weight are carried by the event, whatever they are: what
// kWeightedPairs and WeightedSumsHost do with a Bin outside [0, kBins) and with
// NaN and inf weights.  60 bins: 64 points per CTA in kWeightedPairs.
struct RawWeighted {
    struct Event {
        int32_t bin;
        int32_t pad;
        double w;
    };
    struct Chain {
        double scale;
    };
    static constexpr int kBins = 60;
    __host__ __device__ Chain Prepare(const double* x, int) const {
        Chain c;
        c.scale = x[0];
        return c;
    }
    __host__ __device__ int Bin(const Chain&, const Event& ev) const { return ev.bin; }
    __host__ __device__ double Weight(const Chain& c, const Event& ev) const { return c.scale * ev.w; }
    __host__ __device__ double Finish(const Chain&, const smcmc_user::BinSums& sums, int64_t) const {
        double s = 0.0;
        for (int b = 0; b < kBins; ++b) s = s + (double)(b + 1) * sums[b];
        return s;
    }
};
