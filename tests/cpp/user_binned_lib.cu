// user_binned_lib.cu -- a user translation unit compiled by nvcc into
// libuser_binned.so: it instantiates the binned kernels of smcmc_device_functor.cuh
// for the functors of user_binned.cuh and registers them with engines created by
// anyone (here: Python, through ctypes).  Each engine gets a binding of its own,
// since the count table is used on the engine's stream.
//
//   user_gauss_binned_data(data40)                   the data histogram of later binds
//   user_fake_binned_data(data150, exposure)         the same for FakeBinned
//   user_<name>_bind(engine, events, n, itemsize)    name gauss_binned, fake_binned or raw_binned;
//                                                    0, or -1 with a message for
//                                                    user_binned_error()
//   user_binned_sync(kind, engine, data)             new data histogram, uploaded again
//   user_binned_counts(kind, engine, x, m, dim, out) BinnedBinding::Counts
//   user_binned_host(kind, events, n, x, m, dim, values, counts)
//                                                    BinnedLikelihoodHost / BinnedCountsHost
//   user_fake_binned_events(events, n, out)          FakeBinned::PrepareEvent
// kind: 0 GaussBinned, 1 FakeBinned, 2 RawBinned.
#include <map>
#include <memory>
#include <string>

#include "user_binned.cuh"

static std::string gError;
static GaussBinned gGauss = GaussBinned();
static FakeBinned gFake = FakeBinned();

template <class F>
static std::map<smcmc_engine*, std::unique_ptr<smcmc_user::BinnedBinding<F>>>& Bindings() {
    static std::map<smcmc_engine*, std::unique_ptr<smcmc_user::BinnedBinding<F>>> bindings;
    return bindings;
}
// the functor each engine was bound with, changed by user_binned_sync
template <class F>
static std::map<smcmc_engine*, F>& Functors() {
    static std::map<smcmc_engine*, F> functors;
    return functors;
}

template <class F>
static int BindBinned(smcmc_engine* e, const F& f, const void* events, int64_t n, size_t itemsize) {
    try {
        // the engine keeps its previous binding until the new one is registered
        std::unique_ptr<smcmc_user::BinnedBinding<F>> b(new smcmc_user::BinnedBinding<F>());
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
static int Counts(smcmc_engine* e, const double* x, int m, int dim, uint32_t* out) {
    auto it = Bindings<F>().find(e);
    if (it == Bindings<F>().end()) {
        gError = "no binned functor bound to this engine";
        return -1;
    }
    try {
        it->second->Counts(x, m, dim, out);
        return 0;
    } catch (std::exception& x) {
        gError = x.what();
        return -1;
    }
}

template <class F>
static void Host(const F& f, const void* ev, int64_t n, const double* x, int m, int dim, double* values,
                 uint32_t* counts) {
    const typename F::Event* events = static_cast<const typename F::Event*>(ev);
    for (int p = 0; p < m; ++p) {
        const double* xp = x + (size_t)p * dim;
        if (values) values[p] = smcmc_user::BinnedLikelihoodHost(f, events, n, xp, dim);
        if (counts) smcmc_user::BinnedCountsHost(f, events, n, xp, dim, counts + (size_t)p * F::kBins);
    }
}

// kBinnedPairs' shape without its counting: every counter half set to 1, then the flush.
template <class F>
__global__ void __launch_bounds__(smcmc_user::BinnedShape<F::kBins>::kCtaThreads)
kFlushOnly(int pointTiles, int stride, uint32_t* counts) {
    extern __shared__ __align__(128) unsigned char smem[];
    uint32_t* ctr = reinterpret_cast<uint32_t*>(smem + 2 * smcmc_user::kEventTile * sizeof(typename F::Event));
    for (int w = threadIdx.x; w < F::kBins * 64; w += blockDim.x) ctr[w] = 0x00010001u;
    __syncthreads();
    const int chunk = blockIdx.x / pointTiles;
    smcmc_user::FlushBinCounters<F::kBins>(ctr, counts, stride, (blockIdx.x - chunk * pointTiles) * smcmc_user::kThreads, (int)threadIdx.x);
}

extern "C" {

const char* user_binned_error() { return gError.c_str(); }

void user_gauss_binned_data(const double* data) {
    gGauss.dataTotal = 0.0;
    for (int b = 0; b < GaussBinned::kBins; ++b) {
        gGauss.data[b] = data[b];
        gGauss.dataTotal += data[b];
    }
}
void user_fake_binned_data(const double* data150, double exposure) { gFake.Init(data150, exposure); }

int user_gauss_binned_bind(smcmc_engine* e, const void* ev, int64_t n, size_t itemsize) {
    return BindBinned(e, gGauss, ev, n, itemsize);
}
int user_fake_binned_bind(smcmc_engine* e, const void* ev, int64_t n, size_t itemsize) {
    return BindBinned(e, gFake, ev, n, itemsize);
}
int user_raw_binned_bind(smcmc_engine* e, const void* ev, int64_t n, size_t itemsize) {
    return BindBinned(e, RawBinned(), ev, n, itemsize);
}

// A new data histogram for an engine's functor, uploaded again: SyncLikelihood.
int user_binned_sync(int kind, smcmc_engine* e, const double* data) {
    try {
        if (kind == 0 && Bindings<GaussBinned>().count(e)) {
            GaussBinned& f = Functors<GaussBinned>()[e];
            f.dataTotal = 0.0;
            for (int b = 0; b < GaussBinned::kBins; ++b) {
                f.data[b] = data[b];
                f.dataTotal += data[b];
            }
            Bindings<GaussBinned>()[e]->Upload(f);
            return 0;
        }
        if (kind == 1 && Bindings<FakeBinned>().count(e)) {
            FakeBinned& f = Functors<FakeBinned>()[e];
            for (int k = 0; k < 150; ++k) f.data[k] = data[k];
            Bindings<FakeBinned>()[e]->Upload(f);
            return 0;
        }
    } catch (std::exception& x) {
        gError = x.what();
        return -1;
    }
    gError = "no binned functor of this kind bound to this engine";
    return -1;
}

int user_binned_counts(int kind, smcmc_engine* e, const double* x, int m, int dim, uint32_t* out) {
    if (kind == 0) return Counts<GaussBinned>(e, x, m, dim, out);
    if (kind == 1) return Counts<FakeBinned>(e, x, m, dim, out);
    if (kind == 2) return Counts<RawBinned>(e, x, m, dim, out);
    return -1;
}

// Bind without SetEvents: 1 when it throws std::logic_error, as it must.
int user_gauss_binned_bind_without_sample(smcmc_engine* e) {
    smcmc_user::BinnedBinding<GaussBinned> b;
    try {
        b.Bind(e, gGauss);
    } catch (std::logic_error& x) {
        gError = x.what();
        return 1;
    }
    return 0;
}

int user_binned_host(int kind, const void* ev, int64_t n, const double* x, int m, int dim, double* values,
                     uint32_t* counts) {
    if (kind == 0) Host(gGauss, ev, n, x, m, dim, values, counts);
    else if (kind == 1) Host(gFake, ev, n, x, m, dim, values, counts);
    else if (kind == 2) Host(RawBinned(), ev, n, x, m, dim, values, counts);
    else return -1;
    return 0;
}

int user_fake_binned_events(const smcmc_event* ev, int64_t n, FakeBinned::Event* out) {
    for (int64_t i = 0; i < n; ++i) out[i] = FakeBinned::PrepareEvent(ev[i]);
    return 0;
}

int64_t user_binned_chunk(int64_t n, int64_t pointTiles, int64_t slots) {
    return smcmc_user::BinnedChunk(n, pointTiles, slots);
}

// kBinnedPairs' shape for a kind: threads per CTA, dynamic shared memory, and the
// resident CTAs per SM queried at the first launch of an engine's binding (0 before)
int user_binned_shape(int kind, smcmc_engine* e, int64_t* out3) {
    if (kind == 0) {
        out3[0] = smcmc_user::BinnedBinding<GaussBinned>::kCtaThreads;
        out3[1] = (int64_t)smcmc_user::BinnedBinding<GaussBinned>::kSmemBytes;
        out3[2] = Bindings<GaussBinned>().count(e) ? Bindings<GaussBinned>()[e]->ResidentCtas() : 0;
    } else if (kind == 1) {
        out3[0] = smcmc_user::BinnedBinding<FakeBinned>::kCtaThreads;
        out3[1] = (int64_t)smcmc_user::BinnedBinding<FakeBinned>::kSmemBytes;
        out3[2] = Bindings<FakeBinned>().count(e) ? Bindings<FakeBinned>()[e]->ResidentCtas() : 0;
    } else {
        return -1;
    }
    return 0;
}

// The flush's cost in kBinnedPairs<FakeBinned>: the kernel itself, and a kernel of
// the same shape (threads, shared memory, grid) that only fills the counters so that
// every 16-bit half is non-zero -- the most a flush can have to add -- and runs the
// same FlushBinCounters.  Alternated, `reps` launches each, timed with CUDA events.
// out[0], out[1]: ms per launch of kBinnedPairs and of the flush-only kernel;
// out[2]: resident CTAs per SM; out[3]: CTAs per launch.
int user_fake_binned_flush_time(const void* ev, int64_t n, const double* x, int m, int reps, double* out) {
    typedef FakeBinned F;
    typedef smcmc_user::BinnedBinding<F> B;
    F* df = nullptr;
    F::Event* de = nullptr;
    double* dx = nullptr;
    uint32_t* dc = nullptr;
    const int stride = (m + 31) / 32 * 32;
    const size_t padded = (size_t)((n + smcmc_user::kEventTile - 1) / smcmc_user::kEventTile) * smcmc_user::kEventTile;
    cudaEvent_t t0, t1;
    int dev = 0, sms = 0, resident = 0;
    cudaError_t rc = cudaMalloc((void**)&df, sizeof(F));
    if (!rc) rc = cudaMalloc((void**)&de, padded * sizeof(F::Event));
    if (!rc) rc = cudaMalloc((void**)&dx, (size_t)m * 9 * sizeof(double));
    if (!rc) rc = cudaMalloc((void**)&dc, (size_t)F::kBins * stride * sizeof(uint32_t));
    if (!rc) rc = cudaMemcpy(df, &gFake, sizeof(F), cudaMemcpyHostToDevice);
    if (!rc) rc = cudaMemset(de, 0, padded * sizeof(F::Event));
    if (!rc) rc = cudaMemcpy(de, ev, (size_t)n * sizeof(F::Event), cudaMemcpyHostToDevice);
    if (!rc) rc = cudaMemcpy(dx, x, (size_t)m * 9 * sizeof(double), cudaMemcpyHostToDevice);
    if (!rc) rc = cudaGetDevice(&dev);
    if (!rc) rc = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (!rc) rc = cudaFuncSetAttribute(smcmc_user::kBinnedPairs<F>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)B::kSmemBytes);
    if (!rc) rc = cudaFuncSetAttribute(kFlushOnly<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B::kSmemBytes);
    if (!rc) rc = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, smcmc_user::kBinnedPairs<F>,
                                                                B::kCtaThreads, B::kSmemBytes);
    if (!rc) rc = cudaEventCreate(&t0);
    if (!rc) rc = cudaEventCreate(&t1);
    if (rc) {
        gError = cudaGetErrorString(rc);
        return -1;
    }
    const int pointTiles = (m + smcmc_user::kThreads - 1) / smcmc_user::kThreads;
    const int64_t chunk = smcmc_user::BinnedChunk(n, pointTiles, (int64_t)sms * resident);
    const unsigned grid = (unsigned)((n + chunk - 1) / chunk * pointTiles);
    double ms[2] = {0.0, 0.0};
    for (int r = 0; r <= reps; ++r) {                // r = 0 warms both up
        for (int k = 0; k < 2; ++k) {
            cudaMemsetAsync(dc, 0, (size_t)F::kBins * stride * sizeof(uint32_t));
            cudaEventRecord(t0);
            if (k == 0)
                smcmc_user::kBinnedPairs<F><<<grid, B::kCtaThreads, B::kSmemBytes>>>(df, de, n, (int)chunk, dx, m, 9,
                                                                                  pointTiles, stride, dc);
            else
                kFlushOnly<F><<<grid, B::kCtaThreads, B::kSmemBytes>>>(pointTiles, stride, dc);
            cudaEventRecord(t1);
            cudaEventSynchronize(t1);
            float e = 0.0f;
            cudaEventElapsedTime(&e, t0, t1);
            if (r > 0) ms[k] += e;
        }
    }
    rc = cudaGetLastError();
    cudaEventDestroy(t0);
    cudaEventDestroy(t1);
    cudaFree(df);
    cudaFree(de);
    cudaFree(dx);
    cudaFree(dc);
    if (rc) {
        gError = cudaGetErrorString(rc);
        return -1;
    }
    out[0] = ms[0] / reps;
    out[1] = ms[1] / reps;
    out[2] = resident;
    out[3] = grid;
    return 0;
}

}  // extern "C"
