// user_events_lib.cu -- a user translation unit compiled by nvcc into
// libuser_events.so: it instantiates the event kernels of smcmc_device_functor.cuh
// for the functors of user_events.cuh and registers them with engines created by
// anyone (here: Python, through ctypes).  Each engine gets a binding of its own,
// since the partial-sum scratch is used on the engine's stream.
//
//   user_<name>_bind(engine, events, n, itemsize)    0, or -1 with a message for
//                                                    user_events_error()
//   user_events_host(kind, events, n, x, m, dim, out)  EventLikelihoodHost
#include <map>
#include <memory>
#include <string>

#include "user_events.cuh"

static std::string gError;

template <class F>
static int BindEvents(smcmc_engine* e, const F& f, const void* events, int64_t n, size_t itemsize) {
    static std::map<smcmc_engine*, std::unique_ptr<smcmc_user::EventBinding<F>>> bindings;
    try {
        // the engine keeps its previous binding until the new one is registered
        std::unique_ptr<smcmc_user::EventBinding<F>> b(new smcmc_user::EventBinding<F>());
        b->Bind(e, f, events, n, itemsize);
        bindings[e] = std::move(b);
        return 0;
    } catch (std::exception& x) {
        gError = x.what();
        return -1;
    }
}

static UnbinnedEvents Unbinned() {
    UnbinnedEvents u;
    u.Init();
    return u;
}

extern "C" {

const char* user_events_error() { return gError.c_str(); }

int user_gauss_bind(smcmc_engine* e, const void* ev, int64_t n, size_t itemsize) {
    return BindEvents(e, GaussEvents(), ev, n, itemsize);
}
int user_gauss12_bind(smcmc_engine* e, const void* ev, int64_t n, size_t itemsize) {
    return BindEvents(e, PaddedGaussEvents<Event12>(), ev, n, itemsize);
}
int user_gauss128_bind(smcmc_engine* e, const void* ev, int64_t n, size_t itemsize) {
    return BindEvents(e, PaddedGaussEvents<Event128>(), ev, n, itemsize);
}
int user_unbinned_bind(smcmc_engine* e, const void* ev, int64_t n, size_t itemsize) {
    return BindEvents(e, Unbinned(), ev, n, itemsize);
}

// Bind without SetEvents: 1 when it throws std::logic_error, as it must.
int user_gauss_bind_without_sample(smcmc_engine* e) {
    smcmc_user::EventBinding<GaussEvents> b;
    try {
        b.Bind(e, GaussEvents());
    } catch (std::logic_error& x) {
        gError = x.what();
        return 1;
    }
    return 0;
}

// The chain-local contrast: UnbinnedLoop over a device copy of the events.
int user_unbinned_loop_bind(smcmc_engine* e, const void* ev, int64_t n, size_t itemsize) {
    static std::map<smcmc_engine*, std::unique_ptr<smcmc_user::Binding<UnbinnedLoop>>> bindings;
    static std::map<smcmc_engine*, void*> copies;
    if (itemsize != sizeof(UnbinnedEvents::Event)) {
        gError = "item size";
        return -1;
    }
    if (copies[e]) cudaFree(copies[e]);
    copies[e] = nullptr;
    if (n > 0) {
        if (cudaMalloc(&copies[e], (size_t)n * itemsize) != cudaSuccess ||
            cudaMemcpy(copies[e], ev, (size_t)n * itemsize, cudaMemcpyHostToDevice) != cudaSuccess) {
            gError = "CUDA copy";
            return -1;
        }
    }
    UnbinnedLoop f;
    f.u = Unbinned();
    f.events = (const UnbinnedEvents::Event*)copies[e];
    f.n = n;
    try {
        std::unique_ptr<smcmc_user::Binding<UnbinnedLoop>>& b = bindings[e];
        b.reset(new smcmc_user::Binding<UnbinnedLoop>());
        b->Bind(e, f);
        return 0;
    } catch (std::exception& x) {
        gError = x.what();
        return -1;
    }
}

// kind: 0 GaussEvents, 1 PaddedGaussEvents<Event12>, 2 PaddedGaussEvents<Event128>, 3 UnbinnedEvents
int user_events_host(int kind, const void* ev, int64_t n, const double* x, int m, int dim, double* out) {
    for (int p = 0; p < m; ++p) {
        const double* xp = x + (size_t)p * dim;
        switch (kind) {
        case 0: out[p] = smcmc_user::EventLikelihoodHost(GaussEvents(), (const GaussEvents::Event*)ev, n, xp, dim); break;
        case 1: out[p] = smcmc_user::EventLikelihoodHost(PaddedGaussEvents<Event12>(), (const Event12*)ev, n, xp, dim); break;
        case 2: out[p] = smcmc_user::EventLikelihoodHost(PaddedGaussEvents<Event128>(), (const Event128*)ev, n, xp, dim); break;
        case 3: out[p] = smcmc_user::EventLikelihoodHost(Unbinned(), (const UnbinnedEvents::Event*)ev, n, xp, dim); break;
        default: return -1;
        }
    }
    return 0;
}

int64_t user_event_chunk(int64_t n) { return smcmc_user::EventChunk(n); }
double user_portable_log(double x) { return PortableLog(x); }
int user_event_sizes(int64_t* out) {
    out[0] = sizeof(GaussEvents::Event);
    out[1] = sizeof(Event12);
    out[2] = sizeof(Event128);
    out[3] = sizeof(UnbinnedEvents::Event);
    return 4;
}

}  // extern "C"
