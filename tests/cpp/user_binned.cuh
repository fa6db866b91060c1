// user_binned.cuh -- BINNED event functors written the way a user writes one
// (include/smcmc_device_functor.cuh, "BINNED event functors"): kBinnedPairs and
// kBinnedFinish are instantiated from these types in the translation unit that
// includes this file.
//
//   GaussBinned  a template fit: a standard-normal sample moved to mean x0 and
//                width x1, histogrammed in 40 bins and compared with a data
//                histogram held in the functor by a Poisson likelihood
//   FakeBinned   example/FakeLikelihood.H's histogram fill (the built-in
//                SMCMC_LLH_FAKE, example/ variant) restated as a user functor
//                over events prepared on the host
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>

#include "user_events.cuh"

struct GaussBinned {
    struct Event {
        double z;                 // a standard-normal draw
    };
    struct Chain {
        double mu, sigma;
    };
    static constexpr int kBins = 40;
    static constexpr double kLo = -7.0, kWidth = 0.5;   // bins over [-7, 13)
    double data[kBins];           // the data histogram
    double dataTotal;             // its sum

    __host__ __device__ Chain Prepare(const double* x, int) const {
        Chain c;
        c.mu = x[0];
        c.sigma = x[1];
        return c;
    }
    __host__ __device__ int Bin(const Chain& c, const Event& ev) const {
        const double u = (c.mu + c.sigma * ev.z - kLo) / kWidth;
        if (!(u >= 0.0 && u < (double)kBins)) return -1;
        return (int)floor(u);
    }
    // Poisson log-likelihood (up to a constant) of the data given the template
    // scaled to the data's total, with the reference's floor on an empty bin
    __host__ __device__ double Finish(const Chain&, const smcmc_user::BinCounts& counts, int64_t n) const {
        const double scale = n > 0 ? dataTotal / (double)n : 0.0;
        double s = 0.0;
        for (int b = 0; b < kBins; ++b) {
            double mu = (double)counts[b] * scale;
            if (mu < 0.001) mu = 0.001;
            s = s + (data[b] * PortableLog(mu) - mu);
        }
        return s;
    }
};

// SMCMC_LLH_FAKE (csrc/fake_likelihood.cuh) with the per-event constants prepared
// on the host.  The 300 bins are the built-in's count slots [0, 300):
//   class 0 signal, no decay tag      [  0, 100)  Close bins, then Separated bins
//   class 1 signal, decay tag         [100, 150)  DecayTag bins
//   class 2 background, no decay tag  [150, 250)
//   class 3 background, decay tag     [250, 300)
// Data-typed events (Type < 0) are not binned: the data histogram is in the functor.
struct FakeBinned {
    struct Event {
        double logSigma;          // (log m - log M0) / (log(M0 + S0) - log M0)
        double dLog;              // log m - log M0
        double nomLog;            // log M0
        double sep;               // Separation
        int32_t cls;              // weight class 0..3, -1 for a data-typed event
        int32_t pad;
    };
    struct Chain {
        double skewc, width, scale;
        double sepScale[2];       // signal, background
        double weight[4];         // per class
    };
    static constexpr int kBins = 300;
    // pre-images of the TH1 bin edges under the host's exp: bin of exp(l) is
    // #{k in 1..49 : l >= edges[k]}; the event is cut unless l < edges[50]
    double edges[51];
    double tanFakes, tanEff, pi, exposure;
    double data[150];             // Close, Separated, DecayTag

    // smcmc_event -> Event in SystematicCorrection.H's order, with the host's log
    static Event PrepareEvent(const smcmc_event& e) {
        Event p;
        const double nomLog = std::log(e.TrueMass);
        const double nomLogSigma = std::log(e.TrueMass + e.TrueMassSigma) - nomLog;
        const double d = std::log(e.Mass) - nomLog;
        p.dLog = d;
        p.logSigma = d / nomLogSigma;
        p.nomLog = nomLog;
        p.sep = e.Separation;
        p.cls = e.Type < 0 ? -1 : (e.Type == 0 ? 0 : 2) + (e.MuDk > 0 ? 1 : 0);
        p.pad = 0;
        return p;
    }

    template <class Pred>
    static double FirstLogWhere(Pred pred, double lo, double hi) {
        // bisection over the bit patterns of positive doubles: !pred(exp(lo)), pred(exp(hi))
        uint64_t a, b;
        std::memcpy(&a, &lo, 8);
        std::memcpy(&b, &hi, 8);
        while (b - a > 1) {
            const uint64_t mid = a + (b - a) / 2;
            double m;
            std::memcpy(&m, &mid, 8);
            if (pred(std::exp(m))) b = mid;
            else a = mid;
        }
        double r;
        std::memcpy(&r, &b, 8);
        return r;
    }
    void Init(const double* data150, double exposureRatio) {
        edges[0] = -std::numeric_limits<double>::infinity();
        for (int k = 1; k <= 49; ++k)
            edges[k] = FirstLogWhere([k](double mass) { return 1 + int(50 * (mass - 0.0) / (500.0 - 0.0)) >= k + 1; },
                                     std::log(10.0 * k) - 0.01, std::log(10.0 * k) + 0.01);
        edges[50] = FirstLogWhere([](double mass) { return !(mass < 500.0); }, std::log(500.0) - 0.01,
                                  std::log(500.0) + 0.01);
        tanFakes = std::tan(M_PI * (0.05 - 0.5));
        tanEff = std::tan(M_PI * (0.5 - 0.5));
        pi = M_PI;
        exposure = exposureRatio;
        for (int k = 0; k < 150; ++k) data[k] = data150[k];
    }

    // kFakePrepareChains, example/ variant
    __host__ __device__ Chain Prepare(const double* p, int) const {
        Chain c;
        c.scale = p[2] / 10.0;
        c.width = exp(p[3] / 10.0);
        c.skewc = 0.3 * erf(p[4] / 10.0);
        c.sepScale[0] = exp((0.0 + p[5]) / 10.0);
        c.sepScale[1] = exp((0.0 + p[6]) / 10.0);
        const double wSig = 1.0 * exp(p[0] / 10.0);
        const double wBkg = 1.0 * exp(p[1] / 10.0);
        const double fakes = atan(tanFakes + p[7]) / pi + 0.5;
        const double eff = atan(tanEff + p[8]) / pi + 0.5;
        c.weight[0] = wSig * ((1.0 - fakes) / (1.0 - 0.05)) * exposure;
        c.weight[1] = wSig * (fakes / 0.05) * exposure;
        c.weight[2] = wBkg * ((1.0 - eff) / (1.0 - 0.5)) * exposure;
        c.weight[3] = wBkg * (eff / 0.5) * exposure;
        return c;
    }
    // exactDecide's FP64 sequence, then the separation cut and the class's slot
    __host__ __device__ int Bin(const Chain& c, const Event& ev) const {
        if (ev.cls < 0) return -1;
        const double skew = exp(ev.logSigma * c.skewc);
        double lm = ev.nomLog + ev.dLog * skew;
        lm = ev.nomLog + (lm - ev.nomLog) * c.width;
        lm = lm + c.scale;
        if (!(lm < edges[50])) return -1;                    // above the cut, or NaN
        int k = (int)(expf((float)lm) * 0.1f);               // a guess, corrected below
        k = k < 0 ? 0 : (k > 49 ? 49 : k);
        while (k > 0 && lm < edges[k]) --k;
        while (k < 49 && lm >= edges[k + 1]) ++k;
        const double sep = ev.sep * (ev.cls >> 1 ? c.sepScale[1] : c.sepScale[0]);   // no local-memory index
        if (sep < 0.0) return -1;
        if (!(ev.cls & 1) && !(sep < 100.0)) k += 50;        // the Separated histogram
        const int base = ev.cls == 0 ? 0 : ev.cls == 1 ? 100 : ev.cls == 2 ? 150 : 250;
        return base + k;
    }
    // FakeLikelihood.H:51-59: weights times counts, clamped Poisson term per bin
    __host__ __device__ double Finish(const Chain& c, const smcmc_user::BinCounts& counts, int64_t) const {
        double s = 0.0;
        for (int hb = 0; hb < 150; ++hb) {
            const int h = hb / 50, b = hb - h * 50;
            double mc;
            if (h < 2) mc = c.weight[0] * (double)counts[h * 50 + b] + c.weight[2] * (double)counts[150 + h * 50 + b];
            else mc = c.weight[1] * (double)counts[100 + b] + c.weight[3] * (double)counts[250 + b];
            const double d = data[hb];
            if (mc < 0.001) mc = 0.001;
            double v = d - mc;
            if (d > 0.0) v = v + d * log(mc / d);
            s = s + v;
        }
        return s;
    }
};

// The bin is carried by the event, whatever it is: what kBinnedPairs and
// BinnedCountsHost do with a Bin outside [0, kBins) (negative, kBins, INT_MAX).
// 100 bins: two threads per point in kBinnedPairs.
struct RawBinned {
    struct Event {
        int32_t bin;
        int32_t pad;
    };
    struct Chain {
        double scale;
    };
    static constexpr int kBins = 100;
    __host__ __device__ Chain Prepare(const double* x, int) const {
        Chain c;
        c.scale = x[0];
        return c;
    }
    __host__ __device__ int Bin(const Chain&, const Event& ev) const { return ev.bin; }
    __host__ __device__ double Finish(const Chain& c, const smcmc_user::BinCounts& counts, int64_t) const {
        double s = 0.0;
        for (int b = 0; b < kBins; ++b) s = s + c.scale * (double)(b + 1) * (double)counts[b];
        return s;
    }
};
