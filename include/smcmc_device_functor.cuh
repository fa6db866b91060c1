// smcmc_device_functor.cuh -- user-written likelihood (and gradient) functors
// for the B200 engine: the reference's plugin contract, on the device.
//
// In root-simple-mcmc the whole plugin API is "hand TSimpleMCMC your own
// functor" (reference TSimpleMCMC.H:48-106, :185-187, :544; used that way in
// example/FakeMCMC.C:28-30 and example4/Constrained.C:17-25):
//
//     struct MyLikelihood { double operator()(const sMCMC::Vector& point); };
//     sMCMC::TSimpleMCMC<MyLikelihood> mcmc(tree);
//
// Here the Step hot path runs on the GPU, so the functor's arithmetic has to be
// device code.  A user translation unit compiled by nvcc (-arch=sm_100a)
// includes THIS header (before or instead of TSimpleMCMC.H / TSimpleHMC.H),
// gives the functor a device call operator on a plain array,
//
//     struct MyLikelihood {
//         __host__ __device__ double operator()(const double* x, int n) const;
//         double operator()(const sMCMC::Vector& p) const { return (*this)(p.data(), (int)p.size()); }
//         // optional, for TSimpleHMC<MyLikelihood, MyLikelihood>: the gradient of log L
//         // (reference contract TSimpleHMC.H:38-60: true iff it was computed)
//         __host__ __device__ bool Gradient(const double* x, int n, double* g) const;
//     };
//
// and uses sMCMC::TSimpleMCMC<MyLikelihood> exactly as with the reference header.
// The functor object must be trivially copyable (plain data members, fixed-size
// arrays): it is copied by value to the device, as the reference holds it by
// value (TSimpleMCMC.H:544).  Change its members through GetLogLikelihood() before
// Start(), or call SyncLikelihood() afterwards.
//
// What this header instantiates in the user's translation unit, from the
// functor's type: the evaluation kernels below and two host launch functions,
// registered with the engine as its smcmc_user_ops table entry
// (smcmc_user_set_ops, SMCMC_LLH_USER).  No device function pointer crosses a
// module boundary: libsmcmc_b200.so calls the HOST launch function, which
// queues the kernel compiled here on the engine's stream.
//
// EVENT functors.  A likelihood that is a sum over an event sample (the shape of
// the reference's example/FakeLikelihood.H) is written as a functor with a nested
// Event type and three pieces instead of operator():
//
//     struct MyEvents {
//         struct Event { ... };     // trivially copyable, sizeof <= 128, alignof <= 16
//         struct Chain { ... };     // per-point constants, trivially copyable
//         __host__ __device__ Chain  Prepare(const double* x, int n) const;
//         __host__ __device__ double Term(const Chain& c, const Event& ev) const;
//         // optional (default: return sum)
//         __host__ __device__ double Finish(const Chain& c, double sum, int64_t events) const;
//     };
//     sMCMC::TSimpleMCMC<MyEvents> mcmc;
//     mcmc.SetEvents(events);       // std::vector<MyEvents::Event>, prepared on the host
//
// The value at a point x is Finish(c, S, N) with c = Prepare(x, n) and S the sum of
// Term(c, e) over the N events in this order: the events are cut into chunks of
// EventChunk(N) events in upload order; each chunk sum starts at 0.0 and adds its
// events in order; the chunk sums are added in chunk order, starting at 0.0.  The
// chunk length depends on N alone, so a point's value does not depend on how many
// other points are evaluated with it, on the GPU or on the call, and
// EventLikelihoodHost() restates it on the host.  On the device (kEventPairs) one
// CTA evaluates 128 points, one per thread, over one chunk: the chunk's events are
// staged in shared memory, tile by tile, by TMA bulk copies and read by every
// thread by broadcast.
//
// An event functor has no gradient entry: TSimpleHMC<MyEvents> takes finite
// differences of the likelihood.  A user sample is not split over GPUs: every
// engine of a chain-sharded run holds the whole sample, and the event groups of
// smcmc_comm_init do not reduce a user sum.
//
// BINNED event functors.  A likelihood that fills histograms from the sample and
// compares them with data (a template fit; example/FakeLikelihood.H) is an event
// functor with a bin count and a bin rule instead of Term:
//
//     struct MyBinned {
//         struct Event { ... };     // as for event functors
//         struct Chain { ... };     // per-point constants
//         static constexpr int kBins = 300;                        // 1 <= kBins <= 512
//         __host__ __device__ Chain  Prepare(const double* x, int n) const;
//         __host__ __device__ int    Bin(const Chain& c, const Event& ev) const;   // outside [0, kBins): not counted
//         __host__ __device__ double Finish(const Chain& c, const smcmc_user::BinCounts& counts, int64_t events) const;
//     };
//     sMCMC::TSimpleMCMC<MyBinned> mcmc;  mcmc.SetEvents(events);
//
// It is recognised by F::kBins together with F::Event.  The value at x is
// Finish(c, counts, N) with c = Prepare(x, n) and counts[b] (uint32) the number of
// events with Bin(c, e) == b.  Counts are integers, so they do not depend on how
// the device splits the sample, and BinnedCountsHost() / BinnedLikelihoodHost()
// restate them on the host.  Data histograms live in the functor as fixed-size
// arrays and change as any member does (GetLogLikelihood() before Start(),
// SyncLikelihood() after).  On the device (kBinnedPairs) one CTA counts 128 points
// over one chunk of fewer than 65536 events in private 16-bit shared-memory
// counters and adds them to a global [kBins][points] table; kBinnedFinish applies
// Finish, one thread per point.  A binned likelihood is piecewise constant: it has
// no gradient, and TSimpleHMC refuses it at compile time.
//
// WEIGHTED binned event functors.  A histogram filled with a weight per event and
// per point (Fill(x, w): MC weights, reweighting for systematics) is a binned
// functor with a Weight, and a Finish that receives the weighted sums:
//
//     struct MyWeighted {
//         struct Event { ... };  struct Chain { ... };
//         static constexpr int kBins = 150;                        // 1 <= kBins <= 256
//         __host__ __device__ Chain  Prepare(const double* x, int n) const;
//         __host__ __device__ int    Bin(const Chain& c, const Event& ev) const;      // outside [0, kBins): cut
//         __host__ __device__ double Weight(const Chain& c, const Event& ev) const;   // called for events not cut
//         __host__ __device__ double Finish(const Chain& c, const smcmc_user::BinSums& sums, int64_t events) const;
//     };
//
// It is recognised by F::kBins, F::Event and F::Weight.  The value at x is
// Finish(c, sums, N) with sums[b] the sum of Weight(c, e) over the events with
// Bin(c, e) == b, in this order: the events are cut into chunks of
// WeightedChunk(N) events in upload order; within a chunk each bin's sum starts at
// 0.0 and adds weights in event order; the chunk sums of a bin are added in chunk
// order, starting at 0.0.  So, as for event functors, a point's value does not
// depend on the other points of the call, and WeightedSumsHost() /
// WeightedBinnedLikelihoodHost() restate it on the host.  The weight of a cut
// event is never computed, so a NaN or inf it would have reaches no sum.  On the
// device (kWeightedPairs) each thread keeps one point's FP64 histogram in shared
// memory over one chunk; kWeightedFinish adds the chunks and applies Finish.
// TSimpleHMC refuses it, as it refuses a binned functor.
#ifndef SMCMC_DEVICE_FUNCTOR_CUH_SEEN
#define SMCMC_DEVICE_FUNCTOR_CUH_SEEN

#ifndef __CUDACC__
#error "smcmc_device_functor.cuh must be compiled by nvcc (user device functors are CUDA code)"
#endif

#include <cuda_runtime.h>

#include <cstdint>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <vector>

#include "TSimpleMCMC.H"
#include "smcmc_tma.cuh"

namespace smcmc_user {

constexpr int kThreads = 128;            // points per CTA (one thread per point)
constexpr int kMaxStageBytes = 96 * 1024;

// One THREAD per point.  The kThreads rows of a CTA are one contiguous block of
// the chain-major point array: the CTA copies it to shared memory with coalesced
// loads (row stride ld = n rounded up to odd: lane-per-row reads are then
// conflict-free) and hands every thread a pointer to its own row.  Rows too long
// to stage are read in place.
template <class F>
__global__ void __launch_bounds__(kThreads)
kLikelihood(const F* __restrict__ f, const double* __restrict__ x, int m, int n, int ld, double* __restrict__ out) {
    extern __shared__ double tile[];
    const int base = blockIdx.x * kThreads;
    const int rows = min(kThreads, m - base);
    const int p = base + threadIdx.x;
    if (ld > 0) {
        const double* src = x + (size_t)base * n;
        for (int k = threadIdx.x; k < rows * n; k += kThreads) {
            const int r = k / n;
            tile[r * ld + (k - r * n)] = src[k];
        }
        __syncthreads();
        if (p < m) out[p] = (*f)(tile + threadIdx.x * ld, n);
    } else if (p < m) {
        out[p] = (*f)(x + (size_t)p * n, n);
    }
}

// Gradient of log L at every point that still integrates its trajectory, negated
// (TSimpleHMC.H:478-487: the potential is -log L).  The point and its gradient are
// staged in shared memory when they fit: [rows][ld] points, then [rows][ld] gradients.
template <class F>
__global__ void __launch_bounds__(kThreads)
kGradient(const F* __restrict__ f, const double* __restrict__ x, int m, int n, int ld, double* __restrict__ grad,
          const int32_t* __restrict__ steps, int k) {
    extern __shared__ double tile[];
    const int base = blockIdx.x * kThreads;
    const int rows = min(kThreads, m - base);
    const int p = base + threadIdx.x;
    bool live = p < m;
    if (live && steps) {
        const int s = steps[p];
        live = s >= 1 && k <= s;
    }
    if (ld > 0) {
        double* gt = tile + kThreads * ld;
        const double* src = x + (size_t)base * n;
        for (int q = threadIdx.x; q < rows * n; q += kThreads) {
            const int r = q / n;
            tile[r * ld + (q - r * n)] = src[q];
        }
        __syncthreads();
        bool ok = false;
        if (live) ok = f->Gradient(tile + threadIdx.x * ld, n, gt + threadIdx.x * ld);
        if (live && !ok)
            for (int i = 0; i < n; ++i) gt[threadIdx.x * ld + i] = nan("");   // a functor that declines at run time
        __syncthreads();
        for (int q = threadIdx.x; q < rows * n; q += kThreads) {
            const int r = q / n;
            bool rl = true;
            if (steps) {
                const int s = steps[base + r];
                rl = s >= 1 && k <= s;
            }
            if (rl) grad[(size_t)base * n + q] = -gt[r * ld + (q - r * n)];
        }
    } else if (live) {
        double* g = grad + (size_t)p * n;
        const bool ok = f->Gradient(x + (size_t)p * n, n, g);
        for (int i = 0; i < n; ++i) g[i] = ok ? -g[i] : nan("");
    }
}

template <class F, class = void>
struct HasGradient : std::false_type {};
template <class F>
struct HasGradient<F, decltype((void)std::declval<const F&>().Gradient((const double*)0, 0, (double*)0))> : std::true_type {};

// The device copy of one functor object and its launch table.
template <class F>
class Binding {
    static_assert(std::is_trivially_copyable<F>::value,
                  "a device likelihood functor is copied to the GPU by value: it must be trivially copyable "
                  "(plain data members and fixed-size arrays, no std::vector)");

public:
    Binding() : fDevice(nullptr) {}
    ~Binding() {
        if (fDevice) cudaFree(fDevice);
    }
    Binding(const Binding&) = delete;
    Binding& operator=(const Binding&) = delete;

    /// Copy the functor to the GPU (again).
    void Upload(const F& host) {
        if (!fDevice) Check(cudaMalloc((void**)&fDevice, sizeof(F)));
        Check(cudaMemcpy(fDevice, &host, sizeof(F), cudaMemcpyHostToDevice));
    }
    /// Upload and register with an engine created with SMCMC_LLH_USER.
    void Bind(smcmc_engine* e, const F& host) {
        Upload(host);
        smcmc_user_ops ops;
        ops.struct_size = sizeof ops;
        ops.reserved_ = 0;
        ops.ctx = this;
        ops.likelihood = &Binding::LaunchLikelihood;
        ops.gradient = GradientEntry(HasGradient<F>());
        const int rc = smcmc_user_set_ops(e, &ops);
        if (rc != SMCMC_OK) throw std::logic_error(smcmc_last_error(e));
    }
    static bool kHasGradient() { return HasGradient<F>::value; }

private:
    typedef int (*GradFn)(void*, const double*, int, int, double*, const int32_t*, int, void*);
    static GradFn GradientEntry(std::true_type) { return &Binding::LaunchGradient; }
    static GradFn GradientEntry(std::false_type) { return nullptr; }

    static void Check(cudaError_t rc) {
        if (rc != cudaSuccess) throw std::runtime_error(std::string("CUDA: ") + cudaGetErrorString(rc));
    }
    // shared-memory row stride (0: rows are read in place)
    static int Stride(int n, int copies) {
        const int ld = n | 1;
        return ((size_t)copies * kThreads * ld * sizeof(double) <= (size_t)kMaxStageBytes) ? ld : 0;
    }
    static int LaunchLikelihood(void* ctx, const double* x, int m, int n, double* out, void* stream) {
        Binding* b = static_cast<Binding*>(ctx);
        const int ld = Stride(n, 1);
        const size_t smem = (size_t)kThreads * ld * sizeof(double);
        if (smem > 48 * 1024) {
            cudaError_t rc = cudaFuncSetAttribute(kLikelihood<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (rc != cudaSuccess) return (int)rc;
        }
        kLikelihood<F><<<(m + kThreads - 1) / kThreads, kThreads, smem, (cudaStream_t)stream>>>(b->fDevice, x, m, n, ld, out);
        return (int)cudaGetLastError();
    }
    static int LaunchGradient(void* ctx, const double* x, int m, int n, double* grad, const int32_t* steps, int k,
                              void* stream) {
        Binding* b = static_cast<Binding*>(ctx);
        const int ld = Stride(n, 2);
        const size_t smem = (size_t)2 * kThreads * ld * sizeof(double);
        if (smem > 48 * 1024) {
            cudaError_t rc = cudaFuncSetAttribute(kGradient<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (rc != cudaSuccess) return (int)rc;
        }
        kGradient<F><<<(m + kThreads - 1) / kThreads, kThreads, smem, (cudaStream_t)stream>>>(b->fDevice, x, m, n, ld, grad,
                                                                                            steps, k);
        return (int)cudaGetLastError();
    }

    F* fDevice;
};

// ---------------------------------------------------------------------------
// Event functors
// ---------------------------------------------------------------------------
constexpr int kEventTile = 128;          // events per TMA bulk copy
constexpr int64_t kEventMinChunk = 1024;
constexpr int64_t kEventMaxChunk = 32768;

template <class F, class = void>
struct IsEventFunctor : std::false_type {};
template <class F>
struct IsEventFunctor<F, decltype((void)sizeof(typename F::Event))> : std::true_type {};

template <class F, class = void>
struct HasFinish : std::false_type {};
template <class F>
struct HasFinish<F, decltype((void)std::declval<const F&>().Finish(std::declval<const typename F::Chain&>(), 0.0,
                                                                   (int64_t)0))> : std::true_type {};

template <class F>
struct CheckEventFunctor {
    typedef typename F::Event Event;
    typedef typename F::Chain Chain;
    static_assert(std::is_trivially_copyable<F>::value, "an event functor is copied to the GPU by value: it must be trivially copyable");
    static_assert(std::is_trivially_copyable<Event>::value, "F::Event is copied to the GPU by bytes: it must be trivially copyable");
    static_assert(std::is_trivially_copyable<Chain>::value, "F::Chain must be trivially copyable");
    static_assert(sizeof(Event) <= 128, "sizeof(F::Event) must be at most 128 bytes (a tile of 128 events is staged in shared memory, double buffered)");
    static_assert(alignof(Event) <= 16, "alignof(F::Event) must be at most 16 bytes");
    static constexpr bool value = true;
};

/// Events per chunk of the fixed summation order: about N/256 rounded up to whole
/// tiles, at least kEventMinChunk and at most kEventMaxChunk.  A function of N only.
__host__ __device__ inline int64_t EventChunk(int64_t n) {
    int64_t c = (n + 255) / 256;
    c = (c + kEventTile - 1) / kEventTile * kEventTile;
    return c < kEventMinChunk ? kEventMinChunk : (c > kEventMaxChunk ? kEventMaxChunk : c);
}
__host__ __device__ inline int64_t EventChunks(int64_t n) {
    const int64_t c = EventChunk(n);
    return (n + c - 1) / c;
}

template <class F>
__host__ __device__ inline double EventFinish(const F& f, const typename F::Chain& c, double sum, int64_t n, std::true_type) {
    return f.Finish(c, sum, n);
}
template <class F>
__host__ __device__ inline double EventFinish(const F&, const typename F::Chain&, double sum, int64_t, std::false_type) {
    return sum;
}

/// One CTA = 128 points (one per thread) x one chunk of events.  The chunk is
/// staged tile by tile (kEventTile events, one cp.async.bulk each, double
/// buffered); every thread reads each event of the tile by broadcast and keeps one
/// running sum, written to partial[chunk * stride + point].  The event buffer is
/// padded to whole tiles, so every bulk copy has the same, 16-byte-multiple size.
template <class F>
__global__ void __launch_bounds__(kThreads)
kEventPairs(const F* __restrict__ f, const typename F::Event* __restrict__ events, int64_t n, int chunkEvents,
            const double* __restrict__ x, int m, int dim, int pointTiles, int stride, double* __restrict__ partial) {
    typedef typename F::Event Event;
    constexpr uint32_t kTileBytes = (uint32_t)(kEventTile * sizeof(Event));
    __shared__ __align__(128) Event tiles[2][kEventTile];
    __shared__ __align__(8) uint64_t bars[2];
    const int tid = threadIdx.x;
    const int chunk = blockIdx.x / pointTiles;
    const int point = (blockIdx.x - chunk * pointTiles) * kThreads + tid;
    const int64_t first = (int64_t)chunk * chunkEvents;
    const int count = (int)min((int64_t)chunkEvents, n - first);
    const bool live = point < m;
    typename F::Chain c;
    if (live) c = f->Prepare(x + (size_t)point * dim, dim);

    if (tid == 0) {
        smcmc::mbarInit(&bars[0], 1);
        smcmc::mbarInit(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const Event* src = events + first;
    const int numTiles = (count + kEventTile - 1) / kEventTile;
    if (tid == 0) {
        smcmc::mbarExpectTx(&bars[0], kTileBytes);
        smcmc::tmaLoad1D(tiles[0], src, kTileBytes, &bars[0]);
    }
    double acc = 0.0;
    for (int t = 0; t < numTiles; ++t) {
        const int buf = t & 1;
        if (tid == 0 && t + 1 < numTiles) {
            smcmc::mbarExpectTx(&bars[buf ^ 1], kTileBytes);
            smcmc::tmaLoad1D(tiles[buf ^ 1], src + (size_t)(t + 1) * kEventTile, kTileBytes, &bars[buf ^ 1]);
        }
        smcmc::mbarWait(&bars[buf], (uint32_t)(t >> 1) & 1u);
        const int len = min(kEventTile, count - t * kEventTile);
        if (live) {
#pragma unroll 2
            for (int e = 0; e < len; ++e) acc += f->Term(c, tiles[buf][e]);
        }
        __syncthreads();
    }
    if (live) partial[(size_t)chunk * stride + point] = acc;
}

/// The chunk sums of each point added in chunk order, then Finish.
template <class F>
__global__ void __launch_bounds__(kThreads)
kEventFinish(const F* __restrict__ f, const double* __restrict__ partial, int chunks, int stride, int64_t n,
             const double* __restrict__ x, int m, int dim, double* __restrict__ out) {
    const int p = blockIdx.x * kThreads + threadIdx.x;
    if (p >= m) return;
    double s = 0.0;
    for (int k = 0; k < chunks; ++k) s += partial[(size_t)k * stride + p];
    out[p] = EventFinish(*f, f->Prepare(x + (size_t)p * dim, dim), s, n, HasFinish<F>());
}

/// The value of an event functor at one point, on the host, in the order of the
/// header comment: the reference the device kernels are compared against.
template <class F>
double EventLikelihoodHost(const F& f, const typename F::Event* events, int64_t n, const double* x, int dim) {
    static_assert(CheckEventFunctor<F>::value, "");
    const typename F::Chain c = f.Prepare(x, dim);
    const int64_t chunk = EventChunk(n);
    double s = 0.0;
    for (int64_t first = 0; first < n; first += chunk) {
        const int64_t last = first + chunk < n ? first + chunk : n;
        double part = 0.0;
        for (int64_t i = first; i < last; ++i) part += f.Term(c, events[i]);
        s += part;
    }
    return EventFinish(f, c, s, n, HasFinish<F>());
}

/// The device copy of an event sample, padded with zero bytes to whole tiles so
/// that every bulk copy of the staging loops has the same, 16-byte-multiple size
/// (the padding is never evaluated).  Shared by the event, binned and weighted
/// bindings.
template <class Event>
class EventSample {
public:
    EventSample() : fEvents(nullptr), fCount(-1) {}
    ~EventSample() {
        if (fEvents) cudaFree(fEvents);
    }
    EventSample(const EventSample&) = delete;
    EventSample& operator=(const EventSample&) = delete;

    /// Copy n events to the GPU.  n = 0 is an empty sample.
    void Set(const Event* events, int64_t n) {
        if (n < 0 || (n > 0 && !events)) throw std::invalid_argument("SetEvents: bad event array");
        if (fEvents) Check(cudaFree(fEvents));
        fEvents = nullptr;
        const size_t padded = (size_t)((n + kEventTile - 1) / kEventTile) * kEventTile;
        if (padded > 0) {
            Check(cudaMalloc((void**)&fEvents, padded * sizeof(Event)));
            Check(cudaMemset(fEvents, 0, padded * sizeof(Event)));
            Check(cudaMemcpy(fEvents, events, (size_t)n * sizeof(Event), cudaMemcpyHostToDevice));
        }
        fCount = n;
    }
    bool Has() const { return fCount >= 0; }
    int64_t Count() const { return fCount; }       // -1: no sample set
    const Event* Data() const { return fEvents; }

private:
    static void Check(cudaError_t rc) {
        if (rc != cudaSuccess) throw std::runtime_error(std::string("CUDA: ") + cudaGetErrorString(rc));
    }
    Event* fEvents;
    int64_t fCount;
};

/// The device copies of one event functor and its sample, the partial-sum
/// scratch, and the launch table.  One EventBinding serves one engine (the scratch
/// is used on that engine's stream).
template <class F>
class EventBinding {
    static_assert(CheckEventFunctor<F>::value, "");

public:
    typedef typename F::Event Event;

    EventBinding() : fDevice(nullptr), fPartial(nullptr), fPartialSize(0) {}
    ~EventBinding() {
        if (fDevice) cudaFree(fDevice);
        if (fPartial) cudaFree(fPartial);
    }
    EventBinding(const EventBinding&) = delete;
    EventBinding& operator=(const EventBinding&) = delete;

    /// Copy the sample to the GPU.  n = 0 is an empty sample (sum 0).  Prepare
    /// events on the host before this call.
    void SetEvents(const Event* events, int64_t n) { fSample.Set(events, n); }
    bool HasEvents() const { return fSample.Has(); }
    int64_t GetEventCount() const { return fSample.Count(); }

    /// Copy the functor to the GPU (again).
    void Upload(const F& host) {
        if (!fDevice) Check(cudaMalloc((void**)&fDevice, sizeof(F)));
        Check(cudaMemcpy(fDevice, &host, sizeof(F), cudaMemcpyHostToDevice));
    }
    /// Upload the functor and register with an engine created with SMCMC_LLH_USER;
    /// the sample must have been set.
    void Bind(smcmc_engine* e, const F& host) {
        if (!HasEvents()) throw std::logic_error("event functor: no event sample set (SetEvents) before Bind");
        Upload(host);
        smcmc_user_ops ops;
        ops.struct_size = sizeof ops;
        ops.reserved_ = 0;
        ops.ctx = this;
        ops.likelihood = &EventBinding::LaunchLikelihood;
        ops.gradient = nullptr;                       // finite differences of the likelihood
        const int rc = smcmc_user_set_ops(e, &ops);
        if (rc != SMCMC_OK) throw std::logic_error(smcmc_last_error(e));
    }
    /// Bind with a sample given as raw bytes (a C entry point of a user library):
    /// itemsize must be sizeof(Event).
    void Bind(smcmc_engine* e, const F& host, const void* events, int64_t n, size_t itemsize) {
        if (itemsize != sizeof(Event))
            throw std::invalid_argument("event item size " + std::to_string(itemsize) + " != sizeof(Event) " +
                                        std::to_string(sizeof(Event)));
        SetEvents(static_cast<const Event*>(events), n);
        Bind(e, host);
    }

private:
    static void Check(cudaError_t rc) {
        if (rc != cudaSuccess) throw std::runtime_error(std::string("CUDA: ") + cudaGetErrorString(rc));
    }
    static int LaunchLikelihood(void* ctx, const double* x, int m, int n, double* out, void* stream) {
        EventBinding* b = static_cast<EventBinding*>(ctx);
        cudaStream_t s = (cudaStream_t)stream;
        const int64_t count = b->fSample.Count();
        const int chunks = (int)EventChunks(count);
        const int stride = (m + 31) / 32 * 32;
        const size_t need = (size_t)chunks * stride;
        if (need > b->fPartialSize) {              // grows only: stream-ordered on the engine's stream
            if (b->fPartial) {
                cudaError_t rc = cudaFreeAsync(b->fPartial, s);
                if (rc != cudaSuccess) return (int)rc;
                b->fPartial = nullptr;
                b->fPartialSize = 0;
            }
            cudaError_t rc = cudaMallocAsync((void**)&b->fPartial, need * sizeof(double), s);
            if (rc != cudaSuccess) return (int)rc;
            b->fPartialSize = need;
        }
        const int pointTiles = (m + kThreads - 1) / kThreads;
        if (chunks > 0)
            kEventPairs<F><<<(unsigned)chunks * (unsigned)pointTiles, kThreads, 0, s>>>(
                b->fDevice, b->fSample.Data(), count, (int)EventChunk(count), x, m, n, pointTiles, stride, b->fPartial);
        kEventFinish<F><<<pointTiles, kThreads, 0, s>>>(b->fDevice, b->fPartial, chunks, stride, count, x, m, n, out);
        return (int)cudaGetLastError();
    }

    F* fDevice;
    EventSample<Event> fSample;
    double* fPartial;         // [chunks][stride]
    size_t fPartialSize;
};

// ---------------------------------------------------------------------------
// Binned event functors
// ---------------------------------------------------------------------------
constexpr int kBinnedMaxBins = 512;
// Events per chunk of kBinnedPairs: below 65536, so that a 16-bit counter half
// never carries into its neighbour.
constexpr int64_t kBinnedMaxChunk = 65536 - kEventTile;
static_assert(kBinnedMaxChunk < 65536, "a chunk must not overflow a 16-bit counter");

template <class F, class = void>
struct IsBinnedFunctor : std::false_type {};
template <class F>
struct IsBinnedFunctor<F, decltype((void)F::kBins, (void)sizeof(typename F::Event))> : std::true_type {};

/// counts[b] of one point: a column of the [kBins][stride] count table (stride 1
/// on the host).
class BinCounts {
public:
    __host__ __device__ BinCounts(const uint32_t* first, size_t stride) : fFirst(first), fStride(stride) {}
    __host__ __device__ uint32_t operator[](int b) const { return fFirst[(size_t)b * fStride]; }

private:
    const uint32_t* fFirst;
    size_t fStride;
};

template <class F>
struct CheckBinnedFunctor {
    static_assert(CheckEventFunctor<F>::value, "");
    static_assert(F::kBins >= 1 && F::kBins <= kBinnedMaxBins,
                  "F::kBins must be between 1 and 512 (each bin takes 256 bytes of shared-memory counters per CTA)");
    static_assert(std::is_same<decltype(std::declval<const F&>().Bin(std::declval<const typename F::Chain&>(),
                                                                     std::declval<const typename F::Event&>())),
                               int>::value,
                  "F::Bin(chain, event) must return int");
    static constexpr bool value = true;
};

/// Threads per point of kBinnedPairs: the counters take 256 * kBins bytes per CTA,
/// so fewer CTAs fit an SM as kBins grows; more threads per point keep about 32
/// warps resident (e.g. 300 bins: two CTAs of 512 threads).
template <int Bins>
struct BinnedShape {
    static constexpr int kThreadsPerPoint = Bins <= 96 ? 1 : Bins <= 192 ? 2 : Bins <= 384 ? 4 : 8;
    static constexpr int kCtaThreads = kThreads * kThreadsPerPoint;
};

/// Events per CTA of one kBinnedPairs launch: the grid (chunks x pointTiles) is as
/// close to a whole number of waves of `slots` resident CTAs as whole tiles allow,
/// and a chunk holds at most kBinnedMaxChunk events.  Counts do not depend on it.
inline int64_t BinnedChunk(int64_t n, int64_t pointTiles, int64_t slots) {
    if (pointTiles < 1) pointTiles = 1;
    if (slots < 1) slots = 1;
    const int64_t work = n * pointTiles;
    int64_t waves = (work + slots * kBinnedMaxChunk - 1) / (slots * kBinnedMaxChunk);
    if (waves < 1) waves = 1;
    int64_t c = (work + slots * waves - 1) / (slots * waves);
    c = (c + kEventTile - 1) / kEventTile * kEventTile;
    if (c < kEventTile) c = kEventTile;
    // rounding up the chunk count can spill a few CTAs into one more wave
    while (c < kBinnedMaxChunk && (n + c - 1) / c * pointTiles > slots * waves) c += kEventTile;
    return c > kBinnedMaxChunk ? kBinnedMaxChunk : c;
}

/// The end of a kBinnedPairs chunk: every non-zero 16-bit half of the CTA's
/// counters (word bin * 64 + (p & 63), point p in half p >> 6) is added to
/// counts[bin * stride + base + p] with one global reduction.  All threads of the
/// CTA call it, with their threadIdx.x as tid, after the barrier that ends the
/// counting.
template <int Bins>
__device__ __forceinline__ void FlushBinCounters(const uint32_t* ctr, uint32_t* counts, int stride, int base, int tid) {
    for (int w = tid; w < Bins * 64; w += BinnedShape<Bins>::kCtaThreads) {
        const uint32_t v = ctr[w];
        if (v) {
            uint32_t* dst = counts + (size_t)(w >> 6) * stride + base + (w & 63);
            if (v & 0xffffu) atomicAdd(dst, v & 0xffffu);
            if (v >> 16) atomicAdd(dst + 64, v >> 16);
        }
    }
}

/// One CTA = 128 points x one chunk of events, 128*T threads (T from kBins): thread
/// t takes point t & 127 and every T-th event of each tile.  Tiles are staged as in
/// kEventPairs.  Each point's counters are private to the CTA, in shared memory,
/// 16 bits wide: word bin * 64 + (p & 63) holds point p in half p >> 6, so the 32
/// lanes of a warp (32 consecutive points) hit 32 different banks whatever bins
/// they pick.  An event is counted by one shared-memory atomicAdd of 1 or 1 << 16.
/// At the end of the chunk every non-zero half is added to the global table
/// counts[bin * stride + point].
///
/// The staging loop is kEventPairs' own, not a shared helper: factoring it into
/// one device function changed kEventPairs' SASS (its instruction schedule).
template <class F>
__global__ void __launch_bounds__(BinnedShape<F::kBins>::kCtaThreads)
kBinnedPairs(const F* __restrict__ f, const typename F::Event* __restrict__ events, int64_t n, int chunkEvents,
             const double* __restrict__ x, int m, int dim, int pointTiles, int stride, uint32_t* __restrict__ counts) {
    typedef typename F::Event Event;
    constexpr int T = BinnedShape<F::kBins>::kThreadsPerPoint;
    constexpr int kWords = F::kBins * 64;
    constexpr uint32_t kTileBytes = (uint32_t)(kEventTile * sizeof(Event));
    extern __shared__ __align__(128) unsigned char smem[];
    Event (*tiles)[kEventTile] = reinterpret_cast<Event (*)[kEventTile]>(smem);
    uint32_t* ctr = reinterpret_cast<uint32_t*>(smem + 2 * kTileBytes);
    __shared__ __align__(8) uint64_t bars[2];
    const int tid = threadIdx.x;
    const int lanePoint = tid & (kThreads - 1);
    const int sub = tid / kThreads;
    const int chunk = blockIdx.x / pointTiles;
    const int base = (blockIdx.x - chunk * pointTiles) * kThreads;
    const int point = base + lanePoint;
    const int64_t first = (int64_t)chunk * chunkEvents;
    const int count = (int)min((int64_t)chunkEvents, n - first);
    const bool live = point < m;
    const uint32_t one = lanePoint < 64 ? 1u : (1u << 16);
    uint32_t* mine = ctr + (lanePoint & 63);
    typename F::Chain c;
    if (live) c = f->Prepare(x + (size_t)point * dim, dim);
    for (int w = tid; w < kWords; w += T * kThreads) ctr[w] = 0u;

    if (tid == 0) {
        smcmc::mbarInit(&bars[0], 1);
        smcmc::mbarInit(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const Event* src = events + first;
    const int numTiles = (count + kEventTile - 1) / kEventTile;
    if (tid == 0) {
        smcmc::mbarExpectTx(&bars[0], kTileBytes);
        smcmc::tmaLoad1D(tiles[0], src, kTileBytes, &bars[0]);
    }
    for (int t = 0; t < numTiles; ++t) {
        const int buf = t & 1;
        if (tid == 0 && t + 1 < numTiles) {
            smcmc::mbarExpectTx(&bars[buf ^ 1], kTileBytes);
            smcmc::tmaLoad1D(tiles[buf ^ 1], src + (size_t)(t + 1) * kEventTile, kTileBytes, &bars[buf ^ 1]);
        }
        smcmc::mbarWait(&bars[buf], (uint32_t)(t >> 1) & 1u);
        const int len = min(kEventTile, count - t * kEventTile);
        if (live) {
#pragma unroll 2
            for (int e = sub; e < len; e += T) {
                const int b = f->Bin(c, tiles[buf][e]);
                if ((unsigned)b < (unsigned)F::kBins) atomicAdd(mine + b * 64, one);
            }
        }
        __syncthreads();
    }
    FlushBinCounters<F::kBins>(ctr, counts, stride, base, tid);
}

/// One thread per point: Finish over the point's column of the count table.
template <class F>
__global__ void __launch_bounds__(kThreads)
kBinnedFinish(const F* __restrict__ f, const uint32_t* __restrict__ counts, int stride, int64_t n,
              const double* __restrict__ x, int m, int dim, double* __restrict__ out) {
    const int p = blockIdx.x * kThreads + threadIdx.x;
    if (p >= m) return;
    out[p] = f->Finish(f->Prepare(x + (size_t)p * dim, dim), BinCounts(counts + p, (size_t)stride), n);
}

/// counts[b] = the number of the n events with Bin(Prepare(x), e) == b, on the host.
template <class F>
void BinnedCountsHost(const F& f, const typename F::Event* events, int64_t n, const double* x, int dim,
                      uint32_t* counts) {
    static_assert(CheckBinnedFunctor<F>::value, "");
    const typename F::Chain c = f.Prepare(x, dim);
    for (int b = 0; b < F::kBins; ++b) counts[b] = 0;
    for (int64_t i = 0; i < n; ++i) {
        const int b = f.Bin(c, events[i]);
        if ((unsigned)b < (unsigned)F::kBins) ++counts[b];
    }
}

/// The value of a binned functor at one point, on the host: Finish(c, counts, n).
/// Counts are integers, so the device value equals it whenever Prepare and Finish
/// round alike on the host and the device.
template <class F>
double BinnedLikelihoodHost(const F& f, const typename F::Event* events, int64_t n, const double* x, int dim) {
    std::vector<uint32_t> counts(F::kBins);
    BinnedCountsHost(f, events, n, x, dim, counts.data());
    return f.Finish(f.Prepare(x, dim), BinCounts(counts.data(), 1), n);
}

/// The device copies of one binned functor and its sample, the count table, and
/// the launch table.  One BinnedBinding serves one engine (the table is used on
/// that engine's stream).
template <class F>
class BinnedBinding {
    static_assert(CheckBinnedFunctor<F>::value, "");

public:
    typedef typename F::Event Event;
    static constexpr int kCtaThreads = BinnedShape<F::kBins>::kCtaThreads;
    static constexpr size_t kSmemBytes = 2 * kEventTile * sizeof(Event) + (size_t)F::kBins * 64 * sizeof(uint32_t);

    BinnedBinding() : fDevice(nullptr), fCounts(nullptr), fCountsSize(0), fSlots(0) {}
    ~BinnedBinding() {
        if (fDevice) cudaFree(fDevice);
        if (fCounts) cudaFree(fCounts);
    }
    BinnedBinding(const BinnedBinding&) = delete;
    BinnedBinding& operator=(const BinnedBinding&) = delete;

    /// Copy the sample to the GPU.  n = 0 is an empty sample (all counts 0).
    void SetEvents(const Event* events, int64_t n) { fSample.Set(events, n); }
    bool HasEvents() const { return fSample.Has(); }
    int64_t GetEventCount() const { return fSample.Count(); }

    /// Copy the functor to the GPU (again).
    void Upload(const F& host) {
        if (!fDevice) Check(cudaMalloc((void**)&fDevice, sizeof(F)));
        Check(cudaMemcpy(fDevice, &host, sizeof(F), cudaMemcpyHostToDevice));
    }
    /// Upload the functor and register with an engine created with SMCMC_LLH_USER;
    /// the sample must have been set.
    void Bind(smcmc_engine* e, const F& host) {
        if (!HasEvents()) throw std::logic_error("binned functor: no event sample set (SetEvents) before Bind");
        Upload(host);
        smcmc_user_ops ops;
        ops.struct_size = sizeof ops;
        ops.reserved_ = 0;
        ops.ctx = this;
        ops.likelihood = &BinnedBinding::LaunchLikelihood;
        ops.gradient = nullptr;                       // a binned likelihood is piecewise constant
        const int rc = smcmc_user_set_ops(e, &ops);
        if (rc != SMCMC_OK) throw std::logic_error(smcmc_last_error(e));
    }
    /// Bind with a sample given as raw bytes (a C entry point of a user library):
    /// itemsize must be sizeof(Event).
    void Bind(smcmc_engine* e, const F& host, const void* events, int64_t n, size_t itemsize) {
        if (itemsize != sizeof(Event))
            throw std::invalid_argument("event item size " + std::to_string(itemsize) + " != sizeof(Event) " +
                                        std::to_string(sizeof(Event)));
        SetEvents(static_cast<const Event*>(events), n);
        Bind(e, host);
    }

    /// The counts of the functor last uploaded at m host points x[m][dim]:
    /// out[p * kBins + b], synchronously (the posterior-predictive histogram).
    void Counts(const double* x, int m, int dim, uint32_t* out) {
        if (!HasEvents() || !fDevice) throw std::logic_error("binned functor: Counts before SetEvents and Upload");
        if (m < 1 || dim < 1 || !x || !out) throw std::invalid_argument("Counts: bad point array");
        const int stride = (m + 31) / 32 * 32;
        double* dx = nullptr;
        uint32_t* dc = nullptr;
        std::vector<uint32_t> table((size_t)F::kBins * stride);
        cudaError_t rc = cudaMalloc((void**)&dx, (size_t)m * dim * sizeof(double));
        if (rc == cudaSuccess) rc = cudaMalloc((void**)&dc, table.size() * sizeof(uint32_t));
        if (rc == cudaSuccess) rc = cudaMemcpy(dx, x, (size_t)m * dim * sizeof(double), cudaMemcpyHostToDevice);
        if (rc == cudaSuccess) rc = (cudaError_t)Count(dx, m, dim, dc, stride, 0);
        if (rc == cudaSuccess) rc = cudaMemcpy(table.data(), dc, table.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost);
        if (dx) cudaFree(dx);
        if (dc) cudaFree(dc);
        Check(rc);
        for (int p = 0; p < m; ++p)
            for (int b = 0; b < F::kBins; ++b) out[(size_t)p * F::kBins + b] = table[(size_t)b * stride + p];
    }
    /// Resident CTAs of kBinnedPairs per SM (queried at the first launch; 0 before it).
    int ResidentCtas() const { return fResident; }

private:
    static void Check(cudaError_t rc) {
        if (rc != cudaSuccess) throw std::runtime_error(std::string("CUDA: ") + cudaGetErrorString(rc));
    }
    // clear counts[kBins][stride] and count the sample at m device points, on stream s
    int Count(const double* x, int m, int dim, uint32_t* counts, int stride, cudaStream_t s) {
        const int64_t count = fSample.Count();
        cudaError_t rc = cudaMemsetAsync(counts, 0, (size_t)F::kBins * stride * sizeof(uint32_t), s);
        if (rc != cudaSuccess || count == 0) return (int)rc;
        if (fSlots == 0) {                            // kBinnedPairs' occupancy, once
            int dev = 0, sms = 0;
            if ((rc = cudaGetDevice(&dev)) != cudaSuccess) return (int)rc;
            if ((rc = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return (int)rc;
            if ((rc = cudaFuncSetAttribute(kBinnedPairs<F>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)kSmemBytes)) != cudaSuccess)
                return (int)rc;
            if ((rc = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fResident, kBinnedPairs<F>, kCtaThreads,
                                                                    kSmemBytes)) != cudaSuccess)
                return (int)rc;
            if (fResident < 1) return (int)cudaErrorInvalidConfiguration;
            fSlots = (int64_t)sms * fResident;
        }
        const int pointTiles = (m + kThreads - 1) / kThreads;
        const int64_t chunk = BinnedChunk(count, pointTiles, fSlots);
        if (chunk >= 65536) return (int)cudaErrorInvalidValue;   // a 16-bit counter would overflow
        const int64_t chunks = (count + chunk - 1) / chunk;
        kBinnedPairs<F><<<(unsigned)(chunks * pointTiles), kCtaThreads, kSmemBytes, s>>>(
            fDevice, fSample.Data(), count, (int)chunk, x, m, dim, pointTiles, stride, counts);
        return (int)cudaGetLastError();
    }
    static int LaunchLikelihood(void* ctx, const double* x, int m, int n, double* out, void* stream) {
        BinnedBinding* b = static_cast<BinnedBinding*>(ctx);
        cudaStream_t s = (cudaStream_t)stream;
        const int stride = (m + 31) / 32 * 32;
        const size_t need = (size_t)F::kBins * stride;
        if (need > b->fCountsSize) {                  // grows only: stream-ordered on the engine's stream
            if (b->fCounts) {
                cudaError_t rc = cudaFreeAsync(b->fCounts, s);
                if (rc != cudaSuccess) return (int)rc;
                b->fCounts = nullptr;
                b->fCountsSize = 0;
            }
            cudaError_t rc = cudaMallocAsync((void**)&b->fCounts, need * sizeof(uint32_t), s);
            if (rc != cudaSuccess) return (int)rc;
            b->fCountsSize = need;
        }
        const int rc = b->Count(x, m, n, b->fCounts, stride, s);
        if (rc != (int)cudaSuccess) return rc;
        kBinnedFinish<F><<<(m + kThreads - 1) / kThreads, kThreads, 0, s>>>(b->fDevice, b->fCounts, stride,
                                                                           b->fSample.Count(), x, m, n, out);
        return (int)cudaGetLastError();
    }

    F* fDevice;
    EventSample<Event> fSample;
    uint32_t* fCounts;        // [kBins][stride]
    size_t fCountsSize;
    int64_t fSlots;           // SMs x resident CTAs of kBinnedPairs; 0 until the first launch
    int fResident = 0;
};

// ---------------------------------------------------------------------------
// Weighted binned event functors
// ---------------------------------------------------------------------------
constexpr int kWeightedMaxBins = 256;
constexpr int64_t kWeightedMinChunk = 1024;
constexpr int64_t kWeightedMaxChunks = 32;

template <class F, class = void>
struct IsWeightedBinnedFunctor : std::false_type {};
template <class F>
struct IsWeightedBinnedFunctor<F, decltype((void)F::kBins, (void)sizeof(typename F::Event), (void)&F::Weight)>
    : std::true_type {};

/// sums[b] of one point: a column of a [kBins][stride] table of doubles (stride 1
/// on the host).
class BinSums {
public:
    __host__ __device__ BinSums(const double* first, size_t stride) : fFirst(first), fStride(stride) {}
    __host__ __device__ double operator[](int b) const { return fFirst[(size_t)b * fStride]; }

private:
    const double* fFirst;
    size_t fStride;
};

template <class F>
struct CheckWeightedFunctor {
    static_assert(CheckBinnedFunctor<F>::value, "");
    static_assert(F::kBins >= 1 && F::kBins <= kWeightedMaxBins,
                  "F::kBins of a weighted binned functor must be between 1 and 256 (every point keeps a private "
                  "FP64 histogram in shared memory: 32 points x 256 bins x 8 bytes = 64 KB per CTA)");
    static_assert(std::is_same<decltype(std::declval<const F&>().Weight(std::declval<const typename F::Chain&>(),
                                                                        std::declval<const typename F::Event&>())),
                               double>::value,
                  "F::Weight(chain, event) must return double");
    static constexpr bool value = true;
};

/// Points (= threads) per CTA of kWeightedPairs: 128, 64 or 32, the most whose
/// histograms, Points x kBins doubles, fit 48 KB; 32 above that (up to 64 KB).
template <int Bins>
struct WeightedShape {
    static constexpr int kPoints = Bins * 128 * 8 <= 48 * 1024 ? 128 : Bins * 64 * 8 <= 48 * 1024 ? 64 : 32;
};

/// Events per chunk of the fixed summation order of weighted functors: N/32
/// rounded up to whole tiles, at least kWeightedMinChunk.  A function of N only;
/// a sample is at most kWeightedMaxChunks chunks.
__host__ __device__ inline int64_t WeightedChunk(int64_t n) {
    int64_t c = (n + kWeightedMaxChunks - 1) / kWeightedMaxChunks;
    c = (c + kEventTile - 1) / kEventTile * kEventTile;
    return c < kWeightedMinChunk ? kWeightedMinChunk : c;
}
__host__ __device__ inline int64_t WeightedChunks(int64_t n) {
    const int64_t c = WeightedChunk(n);
    return (n + c - 1) / c;
}

/// One CTA = P points (one thread each, P from kBins) x one chunk of events.  Tiles
/// are staged as in kEventPairs.  Each thread keeps its point's histogram in shared
/// memory, laid out [bin][P] so that a warp's 32 lanes hit consecutive 8-byte
/// words, and adds the weight of every event whose Bin is in [0, kBins) to its bin
/// in event order: a plain load, add and store, no atomics, since no other thread
/// touches the column.  At the end of the chunk the column is written to
/// partial[(chunk * kBins + bin) * stride + point], coalesced across lanes.
///
/// The staging loop is kEventPairs' own, as in kBinnedPairs (§4.10c of DESIGN.md).
template <class F>
__global__ void __launch_bounds__(WeightedShape<F::kBins>::kPoints)
kWeightedPairs(const F* __restrict__ f, const typename F::Event* __restrict__ events, int64_t n, int64_t chunkEvents,
               const double* __restrict__ x, int m, int dim, int pointTiles, int stride, double* __restrict__ partial) {
    typedef typename F::Event Event;
    constexpr int P = WeightedShape<F::kBins>::kPoints;
    constexpr uint32_t kTileBytes = (uint32_t)(kEventTile * sizeof(Event));
    extern __shared__ __align__(128) unsigned char smem[];
    Event (*tiles)[kEventTile] = reinterpret_cast<Event (*)[kEventTile]>(smem);
    __shared__ __align__(8) uint64_t bars[2];
    const int tid = threadIdx.x;
    double* hist = reinterpret_cast<double*>(smem + 2 * kTileBytes) + tid;   // this point's column, stride P
    const int chunk = blockIdx.x / pointTiles;
    const int point = (blockIdx.x - chunk * pointTiles) * P + tid;
    const int64_t first = (int64_t)chunk * chunkEvents;
    const int count = (int)min(chunkEvents, n - first);
    const bool live = point < m;
    typename F::Chain c;
    if (live) c = f->Prepare(x + (size_t)point * dim, dim);
    for (int b = 0; b < F::kBins; ++b) hist[b * P] = 0.0;

    if (tid == 0) {
        smcmc::mbarInit(&bars[0], 1);
        smcmc::mbarInit(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const Event* src = events + first;
    const int numTiles = (count + kEventTile - 1) / kEventTile;
    if (tid == 0) {
        smcmc::mbarExpectTx(&bars[0], kTileBytes);
        smcmc::tmaLoad1D(tiles[0], src, kTileBytes, &bars[0]);
    }
    for (int t = 0; t < numTiles; ++t) {
        const int buf = t & 1;
        if (tid == 0 && t + 1 < numTiles) {
            smcmc::mbarExpectTx(&bars[buf ^ 1], kTileBytes);
            smcmc::tmaLoad1D(tiles[buf ^ 1], src + (size_t)(t + 1) * kEventTile, kTileBytes, &bars[buf ^ 1]);
        }
        smcmc::mbarWait(&bars[buf], (uint32_t)(t >> 1) & 1u);
        const int len = min(kEventTile, count - t * kEventTile);
        if (live) {
#pragma unroll 2
            for (int e = 0; e < len; ++e) {
                const Event& ev = tiles[buf][e];
                const int b = f->Bin(c, ev);
                if ((unsigned)b < (unsigned)F::kBins) hist[b * P] += f->Weight(c, ev);
            }
        }
        __syncthreads();
    }
    if (live)
        for (int b = 0; b < F::kBins; ++b) partial[((size_t)chunk * F::kBins + b) * stride + point] = hist[b * P];
}

/// One thread per point: each bin's chunk partials added in chunk order, starting
/// at 0.0, into the chunk-0 rows (partial[b * stride + point], in place: only this
/// thread reads or writes the column), then Finish over them.  chunks = 0 (an empty
/// sample) leaves every sum 0.0.
template <class F>
__global__ void __launch_bounds__(kThreads)
kWeightedFinish(const F* __restrict__ f, double* __restrict__ partial, int chunks, int stride, int64_t n,
                const double* __restrict__ x, int m, int dim, double* __restrict__ out) {
    const int p = blockIdx.x * kThreads + threadIdx.x;
    if (p >= m) return;
    for (int b = 0; b < F::kBins; ++b) {
        double s = 0.0;
        for (int k = 0; k < chunks; ++k) s += partial[((size_t)k * F::kBins + b) * stride + p];
        partial[(size_t)b * stride + p] = s;
    }
    out[p] = f->Finish(f->Prepare(x + (size_t)p * dim, dim), BinSums(partial + p, (size_t)stride), n);
}

/// sums[b] at one point, on the host, in the order of the header comment: the
/// weights of the events with Bin(c, e) == b, added in event order within each
/// chunk of WeightedChunk(n) events, the chunk sums added in chunk order.
template <class F>
void WeightedSumsHost(const F& f, const typename F::Event* events, int64_t n, const double* x, int dim, double* sums) {
    static_assert(CheckWeightedFunctor<F>::value, "");
    const typename F::Chain c = f.Prepare(x, dim);
    const int64_t chunk = WeightedChunk(n);
    std::vector<double> part(F::kBins);
    for (int b = 0; b < F::kBins; ++b) sums[b] = 0.0;
    for (int64_t first = 0; first < n; first += chunk) {
        const int64_t last = first + chunk < n ? first + chunk : n;
        for (int b = 0; b < F::kBins; ++b) part[b] = 0.0;
        for (int64_t i = first; i < last; ++i) {
            const int b = f.Bin(c, events[i]);
            if ((unsigned)b < (unsigned)F::kBins) part[b] += f.Weight(c, events[i]);
        }
        for (int b = 0; b < F::kBins; ++b) sums[b] += part[b];
    }
}

/// The value of a weighted binned functor at one point, on the host:
/// Finish(c, sums, n) over WeightedSumsHost.
template <class F>
double WeightedBinnedLikelihoodHost(const F& f, const typename F::Event* events, int64_t n, const double* x, int dim) {
    std::vector<double> sums(F::kBins);
    WeightedSumsHost(f, events, n, x, dim, sums.data());
    return f.Finish(f.Prepare(x, dim), BinSums(sums.data(), 1), n);
}

/// The device copies of one weighted binned functor and its sample, the partial
/// sums, and the launch table.  One WeightedBinnedBinding serves one engine (the
/// partial sums are used on that engine's stream).
template <class F>
class WeightedBinnedBinding {
    static_assert(CheckWeightedFunctor<F>::value, "");

public:
    typedef typename F::Event Event;
    static constexpr int kPoints = WeightedShape<F::kBins>::kPoints;
    static constexpr size_t kSmemBytes = 2 * kEventTile * sizeof(Event) + (size_t)F::kBins * kPoints * sizeof(double);

    WeightedBinnedBinding() : fDevice(nullptr), fPartial(nullptr), fPartialSize(0), fResident(0) {}
    ~WeightedBinnedBinding() {
        if (fDevice) cudaFree(fDevice);
        if (fPartial) cudaFree(fPartial);
    }
    WeightedBinnedBinding(const WeightedBinnedBinding&) = delete;
    WeightedBinnedBinding& operator=(const WeightedBinnedBinding&) = delete;

    /// Copy the sample to the GPU.  n = 0 is an empty sample (all sums 0).
    void SetEvents(const Event* events, int64_t n) { fSample.Set(events, n); }
    bool HasEvents() const { return fSample.Has(); }
    int64_t GetEventCount() const { return fSample.Count(); }

    /// Copy the functor to the GPU (again).
    void Upload(const F& host) {
        if (!fDevice) Check(cudaMalloc((void**)&fDevice, sizeof(F)));
        Check(cudaMemcpy(fDevice, &host, sizeof(F), cudaMemcpyHostToDevice));
    }
    /// Upload the functor and register with an engine created with SMCMC_LLH_USER;
    /// the sample must have been set.
    void Bind(smcmc_engine* e, const F& host) {
        if (!HasEvents()) throw std::logic_error("weighted binned functor: no event sample set (SetEvents) before Bind");
        Upload(host);
        smcmc_user_ops ops;
        ops.struct_size = sizeof ops;
        ops.reserved_ = 0;
        ops.ctx = this;
        ops.likelihood = &WeightedBinnedBinding::LaunchLikelihood;
        ops.gradient = nullptr;                       // a binned likelihood is piecewise constant
        const int rc = smcmc_user_set_ops(e, &ops);
        if (rc != SMCMC_OK) throw std::logic_error(smcmc_last_error(e));
    }
    /// Bind with a sample given as raw bytes (a C entry point of a user library):
    /// itemsize must be sizeof(Event).
    void Bind(smcmc_engine* e, const F& host, const void* events, int64_t n, size_t itemsize) {
        if (itemsize != sizeof(Event))
            throw std::invalid_argument("event item size " + std::to_string(itemsize) + " != sizeof(Event) " +
                                        std::to_string(sizeof(Event)));
        SetEvents(static_cast<const Event*>(events), n);
        Bind(e, host);
    }

    /// The weighted histograms of the functor last uploaded at m host points
    /// x[m][dim]: out[p * kBins + b], synchronously, the sums Finish receives.
    void Sums(const double* x, int m, int dim, double* out) {
        if (!HasEvents() || !fDevice) throw std::logic_error("weighted binned functor: Sums before SetEvents and Upload");
        if (m < 1 || dim < 1 || !x || !out) throw std::invalid_argument("Sums: bad point array");
        const int stride = (m + 31) / 32 * 32;
        const size_t need = Scratch(m);
        double* dx = nullptr;
        double* dp = nullptr;
        double* dv = nullptr;
        std::vector<double> table((size_t)F::kBins * stride);
        cudaError_t rc = cudaMalloc((void**)&dx, (size_t)m * dim * sizeof(double));
        if (rc == cudaSuccess) rc = cudaMalloc((void**)&dp, need * sizeof(double));
        if (rc == cudaSuccess) rc = cudaMalloc((void**)&dv, (size_t)m * sizeof(double));
        if (rc == cudaSuccess) rc = cudaMemcpy(dx, x, (size_t)m * dim * sizeof(double), cudaMemcpyHostToDevice);
        if (rc == cudaSuccess) rc = (cudaError_t)Evaluate(dx, m, dim, dp, dv, 0);
        if (rc == cudaSuccess) rc = cudaMemcpy(table.data(), dp, table.size() * sizeof(double), cudaMemcpyDeviceToHost);
        if (dx) cudaFree(dx);
        if (dp) cudaFree(dp);
        if (dv) cudaFree(dv);
        Check(rc);
        for (int p = 0; p < m; ++p)
            for (int b = 0; b < F::kBins; ++b) out[(size_t)p * F::kBins + b] = table[(size_t)b * stride + p];
    }
    /// Resident CTAs of kWeightedPairs per SM (queried at the first launch; 0 before it).
    int ResidentCtas() const { return fResident; }

private:
    static void Check(cudaError_t rc) {
        if (rc != cudaSuccess) throw std::runtime_error(std::string("CUDA: ") + cudaGetErrorString(rc));
    }
    // doubles of partial sums for m points: [max(chunks, 1)][kBins][stride]
    size_t Scratch(int m) const {
        const int64_t chunks = WeightedChunks(fSample.Count());
        return (size_t)(chunks > 1 ? chunks : 1) * F::kBins * (size_t)((m + 31) / 32 * 32);
    }
    // the sums into partial's chunk-0 rows and the values into out, on stream s
    int Evaluate(const double* x, int m, int dim, double* partial, double* out, cudaStream_t s) {
        cudaError_t rc;
        if (fResident == 0) {                         // kWeightedPairs' shared memory and occupancy, once
            if (kSmemBytes > 48 * 1024 &&
                (rc = cudaFuncSetAttribute(kWeightedPairs<F>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)kSmemBytes)) != cudaSuccess)
                return (int)rc;
            if ((rc = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fResident, kWeightedPairs<F>, kPoints,
                                                                    kSmemBytes)) != cudaSuccess)
                return (int)rc;
            if (fResident < 1) return (int)cudaErrorInvalidConfiguration;
        }
        const int64_t n = fSample.Count();
        const int chunks = (int)WeightedChunks(n);
        const int stride = (m + 31) / 32 * 32;
        const int pointTiles = (m + kPoints - 1) / kPoints;
        if (chunks > 0)
            kWeightedPairs<F><<<(unsigned)chunks * (unsigned)pointTiles, kPoints, kSmemBytes, s>>>(
                fDevice, fSample.Data(), n, WeightedChunk(n), x, m, dim, pointTiles, stride, partial);
        kWeightedFinish<F><<<(m + kThreads - 1) / kThreads, kThreads, 0, s>>>(fDevice, partial, chunks, stride, n, x, m,
                                                                             dim, out);
        return (int)cudaGetLastError();
    }
    static int LaunchLikelihood(void* ctx, const double* x, int m, int n, double* out, void* stream) {
        WeightedBinnedBinding* b = static_cast<WeightedBinnedBinding*>(ctx);
        cudaStream_t s = (cudaStream_t)stream;
        const size_t need = b->Scratch(m);
        if (need > b->fPartialSize) {                 // grows only: stream-ordered on the engine's stream
            if (b->fPartial) {
                cudaError_t rc = cudaFreeAsync(b->fPartial, s);
                if (rc != cudaSuccess) return (int)rc;
                b->fPartial = nullptr;
                b->fPartialSize = 0;
            }
            cudaError_t rc = cudaMallocAsync((void**)&b->fPartial, need * sizeof(double), s);
            if (rc != cudaSuccess) return (int)rc;
            b->fPartialSize = need;
        }
        return b->Evaluate(x, m, n, b->fPartial, out, s);
    }

    F* fDevice;
    EventSample<Event> fSample;
    double* fPartial;         // [chunks][kBins][stride]
    size_t fPartialSize;
    int fResident;            // resident CTAs of kWeightedPairs per SM; 0 until the first launch
};

}  // namespace smcmc_user

// The sampler side: a likelihood class WITHOUT a built-in id (no kDeviceLikelihood
// member) is a user device functor; one with a nested Event type is an event functor,
// binned when it also has kBins, weighted binned when it also has Weight.
namespace sMCMC {
namespace detail {
template <class L, class Enable>
struct DeviceBinding {
    static int Kind() { return SMCMC_LLH_USER; }
    static bool HasGradient() { return smcmc_user::HasGradient<L>::value; }
    void Bind(smcmc_engine* e, L& like) { fBinding.Bind(e, like); }
    void Sync(smcmc_engine*, L& like) { fBinding.Upload(like); }
    smcmc_user::Binding<L> fBinding;
};
template <class L, class B>
struct EventSampleBinding {
    typedef typename L::Event Event;
    static int Kind() { return SMCMC_LLH_USER; }
    static bool HasGradient() { return false; }
    void Bind(smcmc_engine* e, L& like) {
        if (fHavePending) {
            fBinding.SetEvents(fPending.data(), (int64_t)fPending.size());
            std::vector<Event>().swap(fPending);
            fHavePending = false;
        }
        fBinding.Bind(e, like);
    }
    void Sync(smcmc_engine*, L& like) { fBinding.Upload(like); }
    // before the engine exists the sample is kept and uploaded by Bind
    void SetEvents(smcmc_engine* e, const std::vector<Event>& events) {
        if (e) {
            fBinding.SetEvents(events.data(), (int64_t)events.size());
        } else {
            fPending = events;
            fHavePending = true;
        }
    }
    std::vector<Event> fPending;
    bool fHavePending = false;
    B fBinding;
};
template <class L>
struct DeviceBinding<L, typename std::enable_if<smcmc_user::IsEventFunctor<L>::value &&
                                                !smcmc_user::IsBinnedFunctor<L>::value>::type>
    : EventSampleBinding<L, smcmc_user::EventBinding<L> > {};
// a binned likelihood is piecewise constant: TSimpleHMC refuses it (kHmcUsable)
template <class L>
struct DeviceBinding<L, typename std::enable_if<smcmc_user::IsBinnedFunctor<L>::value &&
                                                !smcmc_user::IsWeightedBinnedFunctor<L>::value>::type>
    : EventSampleBinding<L, smcmc_user::BinnedBinding<L> > {
    static constexpr bool kHmcUsable = false;
};
template <class L>
struct DeviceBinding<L, typename std::enable_if<smcmc_user::IsWeightedBinnedFunctor<L>::value>::type>
    : EventSampleBinding<L, smcmc_user::WeightedBinnedBinding<L> > {
    static constexpr bool kHmcUsable = false;
};
}  // namespace detail
}  // namespace sMCMC

#endif
