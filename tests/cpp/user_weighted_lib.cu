// user_weighted_lib.cu -- a user translation unit compiled by nvcc into
// libuser_weighted.so: it instantiates the weighted binned kernels of
// smcmc_device_functor.cuh for the functors of user_weighted.cuh and registers
// them with engines created by anyone (here: Python, through ctypes).  Each engine
// gets a binding of its own, since the partial sums are used on the engine's
// stream.
//
//   user_gauss_weighted_data(data40)                   the data histogram of later binds
//   user_fake_weighted_data(data150, exposure)         the same for FakeWeighted
//   user_<name>_bind(engine, events, n, itemsize)      name gauss_weighted, fake_weighted or
//                                                      raw_weighted; 0, or -1 with a message
//                                                      for user_weighted_error()
//   user_weighted_sync(kind, engine, data)             new data histogram, uploaded again
//   user_weighted_sums(kind, engine, x, m, dim, out)   WeightedBinnedBinding::Sums
//   user_weighted_host(kind, events, n, x, m, dim, values, sums)
//                                                      WeightedBinnedLikelihoodHost / WeightedSumsHost
//   user_fake_weighted_events(events, n, out)          FakeWeighted::PrepareEvent
//   user_weighted_chunk(n)                             WeightedChunk
//   user_weighted_shape(kind, engine, out3)            points per CTA, shared memory, resident CTAs
// kind: 0 GaussWeighted, 1 FakeWeighted, 2 RawWeighted.
#include <map>
#include <memory>
#include <string>

#include "user_weighted.cuh"

static std::string gError;
static GaussWeighted gGauss = GaussWeighted();
static FakeWeighted gFake = FakeWeighted();

template <class F>
static std::map<smcmc_engine*, std::unique_ptr<smcmc_user::WeightedBinnedBinding<F>>>& Bindings() {
    static std::map<smcmc_engine*, std::unique_ptr<smcmc_user::WeightedBinnedBinding<F>>> bindings;
    return bindings;
}
// the functor each engine was bound with, changed by user_weighted_sync
template <class F>
static std::map<smcmc_engine*, F>& Functors() {
    static std::map<smcmc_engine*, F> functors;
    return functors;
}

template <class F>
static int BindWeighted(smcmc_engine* e, const F& f, const void* events, int64_t n, size_t itemsize) {
    try {
        // the engine keeps its previous binding until the new one is registered
        std::unique_ptr<smcmc_user::WeightedBinnedBinding<F>> b(new smcmc_user::WeightedBinnedBinding<F>());
        b->Bind(e, f, events, n, itemsize);
        Bindings<F>()[e] = std::move(b);
        Functors<F>()[e] = f;
        return 0;
    } catch (std::exception& x) {
        gError = x.what();
        return -1;
    }
}

template <class F>
static int Sums(smcmc_engine* e, const double* x, int m, int dim, double* out) {
    auto it = Bindings<F>().find(e);
    if (it == Bindings<F>().end()) {
        gError = "no weighted binned functor bound to this engine";
        return -1;
    }
    try {
        it->second->Sums(x, m, dim, out);
        return 0;
    } catch (std::exception& x) {
        gError = x.what();
        return -1;
    }
}

template <class F>
static void Host(const F& f, const void* ev, int64_t n, const double* x, int m, int dim, double* values, double* sums) {
    const typename F::Event* events = static_cast<const typename F::Event*>(ev);
    for (int p = 0; p < m; ++p) {
        const double* xp = x + (size_t)p * dim;
        if (values) values[p] = smcmc_user::WeightedBinnedLikelihoodHost(f, events, n, xp, dim);
        if (sums) smcmc_user::WeightedSumsHost(f, events, n, xp, dim, sums + (size_t)p * F::kBins);
    }
}

template <class F>
static void Shape(smcmc_engine* e, int64_t* out3) {
    out3[0] = smcmc_user::WeightedBinnedBinding<F>::kPoints;
    out3[1] = (int64_t)smcmc_user::WeightedBinnedBinding<F>::kSmemBytes;
    out3[2] = Bindings<F>().count(e) ? Bindings<F>()[e]->ResidentCtas() : 0;
}

static void SetGaussData(GaussWeighted& f, const double* data) {
    f.dataTotal = 0.0;
    for (int b = 0; b < GaussWeighted::kBins; ++b) {
        f.data[b] = data[b];
        f.dataTotal += data[b];
    }
}

extern "C" {

const char* user_weighted_error() { return gError.c_str(); }

void user_gauss_weighted_data(const double* data) { SetGaussData(gGauss, data); }
void user_fake_weighted_data(const double* data150, double exposure) { gFake.Init(data150, exposure); }

int user_gauss_weighted_bind(smcmc_engine* e, const void* ev, int64_t n, size_t itemsize) {
    return BindWeighted(e, gGauss, ev, n, itemsize);
}
int user_fake_weighted_bind(smcmc_engine* e, const void* ev, int64_t n, size_t itemsize) {
    return BindWeighted(e, gFake, ev, n, itemsize);
}
int user_raw_weighted_bind(smcmc_engine* e, const void* ev, int64_t n, size_t itemsize) {
    return BindWeighted(e, RawWeighted(), ev, n, itemsize);
}

// A new data histogram for an engine's functor, uploaded again: SyncLikelihood.
int user_weighted_sync(int kind, smcmc_engine* e, const double* data) {
    try {
        if (kind == 0 && Bindings<GaussWeighted>().count(e)) {
            GaussWeighted& f = Functors<GaussWeighted>()[e];
            SetGaussData(f, data);
            Bindings<GaussWeighted>()[e]->Upload(f);
            return 0;
        }
        if (kind == 1 && Bindings<FakeWeighted>().count(e)) {
            FakeWeighted& f = Functors<FakeWeighted>()[e];
            for (int k = 0; k < 150; ++k) f.fake.data[k] = data[k];
            Bindings<FakeWeighted>()[e]->Upload(f);
            return 0;
        }
    } catch (std::exception& x) {
        gError = x.what();
        return -1;
    }
    gError = "no weighted binned functor of this kind bound to this engine";
    return -1;
}

int user_weighted_sums(int kind, smcmc_engine* e, const double* x, int m, int dim, double* out) {
    if (kind == 0) return Sums<GaussWeighted>(e, x, m, dim, out);
    if (kind == 1) return Sums<FakeWeighted>(e, x, m, dim, out);
    if (kind == 2) return Sums<RawWeighted>(e, x, m, dim, out);
    return -1;
}

// Bind without SetEvents: 1 when it throws std::logic_error, as it must.
int user_gauss_weighted_bind_without_sample(smcmc_engine* e) {
    smcmc_user::WeightedBinnedBinding<GaussWeighted> b;
    try {
        b.Bind(e, gGauss);
    } catch (std::logic_error& x) {
        gError = x.what();
        return 1;
    }
    return 0;
}

int user_weighted_host(int kind, const void* ev, int64_t n, const double* x, int m, int dim, double* values,
                       double* sums) {
    if (kind == 0) Host(gGauss, ev, n, x, m, dim, values, sums);
    else if (kind == 1) Host(gFake, ev, n, x, m, dim, values, sums);
    else if (kind == 2) Host(RawWeighted(), ev, n, x, m, dim, values, sums);
    else return -1;
    return 0;
}

int user_fake_weighted_events(const smcmc_event* ev, int64_t n, FakeWeighted::Event* out) {
    for (int64_t i = 0; i < n; ++i) out[i] = FakeWeighted::PrepareEvent(ev[i]);
    return 0;
}

int64_t user_weighted_chunk(int64_t n) { return smcmc_user::WeightedChunk(n); }

// kWeightedPairs' shape for a kind: points (threads) per CTA, dynamic shared memory,
// and the resident CTAs per SM queried at the first launch of an engine's binding
// (0 before)
int user_weighted_shape(int kind, smcmc_engine* e, int64_t* out3) {
    if (kind == 0) Shape<GaussWeighted>(e, out3);
    else if (kind == 1) Shape<FakeWeighted>(e, out3);
    else if (kind == 2) Shape<RawWeighted>(e, out3);
    else return -1;
    return 0;
}

}  // extern "C"
