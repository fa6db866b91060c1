/* smcmc_b200.h -- C ABI of libsmcmc_b200.so, the B200 (sm_100a) ensemble
 * Metropolis engine that sits behind the root-simple-mcmc header API.
 *
 * One engine handle owns, on one GPU, the device state of `chains`
 * independent Markov chains of dimension `dim`:  the state that ONE
 * sMCMC::TSimpleMCMC<L, TProposeAdaptiveStep> object holds on the host in the
 * reference (TSimpleMCMC.H:543-589 and :1833-1976), replicated per chain.
 * Every entry point below names the reference interface it replaces.  All
 * pointers are HOST pointers unless a name ends in _dev; all functions return
 * 0 on success and a negative smcmc_status otherwise, with a message
 * available from smcmc_last_error().  A handle is not thread-safe; use one
 * host thread per handle.  There is no CPU fallback: creating an engine
 * without a CUDA device fails.
 *
 * Random draws: chain c (global index chain_offset + c) at step s uses slots
 * 0..dim of the counter-based stream defined in smcmc_rng.h.
 */
#ifndef SMCMC_B200_H_SEEN
#define SMCMC_B200_H_SEEN

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMCMC_B200_ABI_VERSION 2

typedef struct smcmc_engine smcmc_engine;

typedef enum smcmc_status {
    SMCMC_OK = 0,
    SMCMC_ERR_INVALID_ARGUMENT = -1, /* std::invalid_argument in the reference */
    SMCMC_ERR_LOGIC = -2,            /* std::logic_error                      */
    SMCMC_ERR_RUNTIME = -3,          /* std::runtime_error                    */
    SMCMC_ERR_CUDA = -4,             /* CUDA runtime failure                  */
    SMCMC_ERR_NO_DEVICE = -5         /* no usable sm_100 device               */
} smcmc_status;

/* Built-in device likelihood functors (SURVEY.md 8a rows a5-a8). */
typedef enum smcmc_likelihood {
    SMCMC_LLH_UNIT_GAUSS = 0, /* -1/2 sum x^2        TSimpleMCMC.H:111-120        */
    SMCMC_LLH_DUMMY = 1,      /* -1/2 x^T E x        TDummyLogLikelihood.H:21-31  */
    SMCMC_LLH_HORRIFIC = 2,   /* box + ridge         THorrificLogLikelihood.H:26-38 */
    SMCMC_LLH_ASYM = 3,       /* piecewise linear    TAsymLogLikelihood.H:20-31   */
    SMCMC_LLH_FAKE = 4,       /* event reweighting + binned Poisson,
                                 example/FakeLikelihood.H:47-81,188-216          */
    SMCMC_LLH_UNBINNED = 5,   /* NOT in the reference: unbinned mixture likelihood over
                                 events (BASELINE.json configs[4]); see
                                 smcmc_unbinned_set_events                        */
    SMCMC_LLH_HARD = 6,       /* Rosenbrock valley   THardLogLikelihood.H:57-91 (with its
                                 gradient functor for TSimpleHMC), dim >= 2       */
    SMCMC_LLH_FAKE2 = 7,      /* example2/FakeLikelihood.H:58-118,222-289: the same event
                                 corrections and cuts, signal and background filled into
                                 separate histograms, each renormalised to the event
                                 counts x[0], x[1] by its integral, plus the penalty terms
                                 (:91-115).  Events and data histograms are set with the
                                 smcmc_fake_* calls; the exposure argument is not used  */
    SMCMC_LLH_USER = 8        /* a USER-WRITTEN device functor: the reference's plugin contract
                                 (TSimpleMCMC.H:48-106: "hand TSimpleMCMC your own functor",
                                 used that way in example/FakeMCMC.C:28-30 and
                                 example4/Constrained.C:17-25).  The functor is compiled by nvcc
                                 in the user's translation unit together with the kernel
                                 templates of include/smcmc_device_functor.cuh and registered
                                 with smcmc_user_set_ops; any dimension                        */
} smcmc_likelihood;

/* The table entry of a user device functor (SMCMC_LLH_USER).  Both entries are HOST
 * functions of the user's translation unit that queue a kernel on `cuda_stream`
 * (include/smcmc_device_functor.cuh instantiates them from the functor's type);
 * pointers ending in _dev are device pointers.  They return 0 or a cudaError_t. */
typedef struct smcmc_user_ops {
    uint32_t struct_size;   /* sizeof(smcmc_user_ops)                                          */
    uint32_t reserved_;
    void* ctx;              /* passed back to the two functions                                */
    /* UserLikelihood::operator() (TSimpleMCMC.H:59-69) at m points: x_dev[m*dim] -> llh_dev[m] */
    int (*likelihood)(void* ctx, const double* x_dev, int m, int dim, double* llh_dev, void* cuda_stream);
    /* UserGradient::operator() (TSimpleHMC.H:38-60, called at :478-487): the gradient of
     * log L at the m points, NEGATED into grad_dev[m*dim] (the potential's gradient, :486).
     * Chain c takes part when steps_dev == NULL or 1 <= steps_dev[c] and k <= steps_dev[c]
     * (chains of an ensemble carry their own trajectory length).  NULL: the functor has no
     * gradient (TSimpleHMC<L>: finite differences, :417-444).                                 */
    int (*gradient)(void* ctx, const double* x_dev, int m, int dim, double* grad_dev,
                    const int32_t* steps_dev, int k, void* cuda_stream);
} smcmc_user_ops;

typedef struct smcmc_config {
    uint32_t struct_size;   /* sizeof(smcmc_config), for ABI growth            */
    int32_t device;         /* CUDA device ordinal                             */
    int32_t dim;            /* parameters per chain                            */
    int32_t chains;         /* chains owned by this engine (this GPU's shard)  */
    uint32_t chain_offset;  /* global index of local chain 0 (RNG addressing)  */
    int32_t likelihood;     /* smcmc_likelihood                                */
    uint64_t seed;          /* run seed (Philox key)                           */
} smcmc_config;

/* The reference's MC event record, example/Simulated.H:7-14, 48 bytes. */
typedef struct smcmc_event {
    double Mass;
    int32_t Type;           /* 0 signal, >0 background, <0 data                */
    int32_t pad0_;
    double Separation;
    int32_t MuDk;
    int32_t pad1_;
    double TrueMass;
    double TrueMassSigma;
} smcmc_event;

/* Scalar settings of the adaptive proposal; each names the
 * TProposeAdaptiveStep setter (TSimpleMCMC.H line) it stands for.  Settings
 * apply to every chain of the engine. */
typedef enum smcmc_prop_field {
    SMCMC_PROP_SIGMA = 0,                /* SetSigma                       :775  */
    SMCMC_PROP_TARGET_ACCEPTANCE = 1,    /* SetTargetAcceptance            :977  */
    SMCMC_PROP_ACCEPTANCE_WINDOW = 2,    /* SetAcceptanceWindow            :982  */
    SMCMC_PROP_ACCEPTANCE_RIGIDITY = 3,  /* SetAcceptanceRigidity          :1002 */
    SMCMC_PROP_ACCEPTANCE_DEWEIGHT = 4,  /* SetAcceptanceUpdateDeweighting :987  */
    SMCMC_PROP_COVARIANCE_WINDOW = 5,    /* SetCovarianceWindow            :914  */
    SMCMC_PROP_COVARIANCE_DEWEIGHT = 6,  /* SetCovarianceUpdateDeweighting :927  */
    SMCMC_PROP_COVARIANCE_FROZEN = 7,    /* SetCovarianceFrozen            :937  */
    SMCMC_PROP_COVARIANCE_TRIALS = 8,    /* SetCovarianceTrials            :947  */
    SMCMC_PROP_CENTER_TRIALS = 9,        /* SetEstimatedCenterTrials       :747  */
    SMCMC_PROP_NEXT_UPDATE = 10,         /* SetNextUpdate                  :992  */
    SMCMC_PROP_MAX_CORRELATION = 11,     /* SetMaximumCorrelation          :909  */
    SMCMC_PROP_STEP_RMS_WINDOW = 12,     /* TSimpleMCMC::SetStepRMSWindow  :511  */
    SMCMC_PROP_POOLED_EVERY = 13,        /* NEW (not in the reference): K > 0 pools the
                                            covariance adaptation over all chains and
                                            GPUs, exchanging statistics every K steps   */
    SMCMC_PROP_KIND = 15,                /* which proposal functor the sampler is instantiated with
                                            (smcmc_proposal_kind); before smcmc_start          */
    SMCMC_PROP_POOLED_TENSOR = 14        /* pooled mode: evaluate x' = x + (sigma z).U of all
                                            chains as one GEMM on the FP64 tensor cores;
                                            -1 automatic (dim >= 128, default), 0 off, 1 on */
} smcmc_prop_field;

/* Per-chain quantities readable with smcmc_get().  Arrays are chain-major:
 * element (c, i) at [c*dim + i]; packed covariance is lower-triangular
 * row-major exactly as the AdaptiveCovariance branch (TSimpleMCMC.H:1645-1649).
 */
typedef enum smcmc_field {
    SMCMC_F_ACCEPTED = 0,        /* double[chains*dim]   GetAccepted              :502 */
    SMCMC_F_PROPOSED = 1,        /* double[chains*dim]   GetProposed              :514 */
    SMCMC_F_ACCEPTED_LLH = 2,    /* double[chains]       GetAcceptedLogLikelihood :499 */
    SMCMC_F_PROPOSED_LLH = 3,    /* double[chains]       GetProposedLogLikelihood :505 */
    SMCMC_F_STEP_RMS = 4,        /* double[chains]       GetStepRMS               :508 */
    SMCMC_F_SIGMA = 5,           /* double[chains]       GetSigma                 :770 */
    SMCMC_F_ACCEPTANCE = 6,      /* double[chains]       GetAcceptance            :781 */
    SMCMC_F_ACCEPTANCE_TRIALS = 7, /* double[chains]     GetAcceptanceTrials      :782 */
    SMCMC_F_ACCEPTANCE_RIGIDITY = 8, /* double[chains]   GetAcceptanceRigidity    :1003 */
    SMCMC_F_TRIALS = 9,          /* int32[chains]        GetTrials                :762 */
    SMCMC_F_SUCCESSES = 10,      /* int32[chains]        GetSuccesses             :765 */
    SMCMC_F_NEXT_UPDATE = 11,    /* int32[chains]        GetNextUpdate            :993 */
    SMCMC_F_COVARIANCE_TRIALS = 12, /* double[chains]    GetCovarianceTrials      :942 */
    SMCMC_F_CENTER_TRIALS = 13,  /* double[chains]       GetEstimatedCenterTrials :741 */
    SMCMC_F_CENTER = 14,         /* double[chains*dim]   GetEstimatedCenter       :732 */
    SMCMC_F_COVARIANCE = 15,     /* double[chains*dim*(dim+1)/2] packed           */
    SMCMC_F_COVARIANCE_TRACE = 16, /* double[chains]     GetCovarianceTrace       :961 */
    SMCMC_F_DECOMPOSITION = 17,  /* double[chains*dim*dim] row-major U, fDecomposition :1893 */
    SMCMC_F_TOTAL_STEPS = 18,    /* int32[chains]        fTotalSteps              :554 */
    SMCMC_F_LLH_CALLS = 19,      /* int32[chains]        GetLogLikelihoodCount    :242 */
    SMCMC_F_STATUS = 20,         /* int32[chains]        0 ok, else smcmc_status of the
                                    exception the reference would have thrown    */
    SMCMC_F_SIGMA_TRACE = 21,    /* double[chains]       fSigmaTrace              :1960 */
    SMCMC_F_COVARIANCE_WINDOW = 22, /* double[1]         GetCovarianceWindow      :915 */
    SMCMC_F_ACCEPTANCE_WINDOW = 23, /* double[1]         GetAcceptanceWindow      :983 */
    SMCMC_F_TARGET_ACCEPTANCE = 24, /* double[1]         GetTargetAcceptance      :978 */
    SMCMC_F_POOLED_MEAN = 25,       /* double[dim]       pooled mode: ensemble mean        */
    SMCMC_F_POOLED_COVARIANCE = 26, /* double[dim*(dim+1)/2] pooled mode: packed covariance */
    SMCMC_F_POOLED_DECOMPOSITION = 27, /* double[dim*dim] pooled mode: the shared U         */
    SMCMC_F_POOLED_COUNT = 28,      /* double[1]         points behind the pooled estimate */
    /* TProposeVAATStep (SMCMC_PROPOSAL_VAAT); with it SMCMC_F_SIGMA and SMCMC_F_ACCEPTANCE are
     * its GetSigma / GetAcceptance: the means over the dimensions (TProposeVAATStep.H:155-173) */
    SMCMC_F_VAAT_SIGMA = 29,        /* double[chains*dim] fSigma            :299 */
    SMCMC_F_VAAT_ACCEPTANCE = 30,   /* double[chains*dim] fAcceptance       :290 */
    SMCMC_F_VAAT_ACCEPTANCE_TRIALS = 31, /* int32[chains*dim] fAcceptanceTrials :293 */
    SMCMC_F_VAAT_LAST_INDEX = 32,   /* int32[chains]      fLastIndex        :275 */
    SMCMC_F_VAAT_QUEUE = 33         /* int32[chains]      indices left in fNextIndex :272 */
} smcmc_field;

/* The proposal functor of the sampler (SMCMC_PROP_KIND). */
typedef enum smcmc_proposal_kind {
    SMCMC_PROPOSAL_ADAPTIVE = 0,    /* sMCMC::TProposeAdaptiveStep, TSimpleMCMC.H:640-1977 (default;
                                       TProposeSimpleStep is this one with its adaptation frozen)   */
    SMCMC_PROPOSAL_VAAT = 1         /* sMCMC::TProposeVAATStep, TProposeVAATStep.H:22-307: adaptive
                                       variable-at-a-time.  Settings that exist for it: SetGaussian
                                       (sigma itself), SetUniform, SetAcceptanceWindow (reset to 100
                                       by the first Start, as in the reference), SetAcceptanceRigidity;
                                       no save / restore (the reference's returns false)            */
} smcmc_proposal_kind;

/* Optional per-step trace of smcmc_step_trace(); any pointer may be NULL.
 * Step-major: entry (s, c) at [s*chains + c], points at [(s*chains+c)*dim]. */
typedef struct smcmc_trace {
    int32_t* accepted;      /* return value of TSimpleMCMC::Step  :370 */
    double* llh_accepted;   /* LogLikelihood branch               :208 */
    double* llh_proposed;
    double* points;         /* Accepted branch                    :210 */
    double* sigma;          /* AdaptiveSigma branch               :1621 */
    double* step_rms;       /* StepRMS branch                     :211 */
} smcmc_trace;

int smcmc_abi_version(void);

/* Global (handle-less) error text of the last failed smcmc_create. */
const char* smcmc_last_error(const smcmc_engine* e);

/* TSimpleMCMC(TTree*, bool) constructor, TSimpleMCMC.H:203-224, for `chains`
 * chains at once.  Allocates all device state. */
int smcmc_create(const smcmc_config* cfg, smcmc_engine** out);
int smcmc_destroy(smcmc_engine* e);

/* Launch on the caller's CUDA stream (a cudaStream_t); NULL = default. */
int smcmc_set_stream(smcmc_engine* e, void* cuda_stream);
/* Block until all queued work is done; reports asynchronous errors. */
int smcmc_sync(smcmc_engine* e);

/* ---- multi-GPU: NCCL over NVLink (one engine = one rank = one GPU) --------- */
/* Rank 0 creates the 128-byte NCCL unique id and distributes it out of band. */
int smcmc_comm_unique_id(char* out, size_t bytes);
/* Join `world` ranks.  Ranks [k*event_group, (k+1)*event_group) form an EVENT
 * GROUP: they must be created with the same chains / chain_offset / seed, each
 * uploads its own slice of the events, and every likelihood evaluation
 * all-reduces the integer event counts inside the group.  The world
 * communicator all-reduces the pooled adaptation statistics
 * (SMCMC_PROP_POOLED_EVERY).  Chain-sharded ensembles with per-chain adaptation
 * need no communicator at all. */
int smcmc_comm_init(smcmc_engine* e, const char* unique_id, size_t bytes, int world, int rank,
                    int event_group);

/* ---- proposal configuration: TProposeAdaptiveStep setters ---------------- */
int smcmc_prop_set(smcmc_engine* e, int field, double value);
int smcmc_prop_set_gaussian(smcmc_engine* e, int dim, double sigma);      /* :855 */
int smcmc_prop_set_uniform(smcmc_engine* e, int dim, double lo, double hi); /* :833 */
int smcmc_prop_set_correlation(smcmc_engine* e, int d1, int d2, double c);  /* :883 */
int smcmc_prop_reset_correlations(smcmc_engine* e);                       /* :874 */
int smcmc_prop_update(smcmc_engine* e);   /* UpdateProposal() on every chain :1009 */
int smcmc_prop_reset(smcmc_engine* e);    /* ResetProposal()  on every chain :1396 */

/* Debugging modes of the proposal functor (TSimpleMCMC.H:671-704).
 * ForceStep (:811-818): the NEXT step proposes the given point (x[dim] for every chain,
 * or x[chains*dim] with per_chain != 0) without touching the adaptive state; combine
 * with metropolis = 2 to move the chains there (the idiom of :797-808). */
int smcmc_prop_force_step(smcmc_engine* e, const double* x, int per_chain);
/* SetScanDimension (:820-830): while dim is a valid dimension every step only redraws
 * that coordinate around the estimated centre (one draw); -1 (or out of range) = off. */
int smcmc_prop_set_scan_dimension(smcmc_engine* e, int dim);
/* SetEstimatedCenter (:733-739): v[dim] for every chain, or v[chains*dim]. */
int smcmc_prop_set_center(smcmc_engine* e, const double* v, int per_chain);

/* ---- likelihood inputs --------------------------------------------------- */
/* SMCMC_LLH_USER: register the functor's launch table; before smcmc_start. */
int smcmc_user_set_ops(smcmc_engine* e, const smcmc_user_ops* ops);
/* FakeLikelihood::SimulatedSample (example/FakeLikelihood.H:30); events are
 * copied to the device and re-laid-out there.  Replaces the sample. */
int smcmc_fake_set_events(smcmc_engine* e, const smcmc_event* events, int64_t n);
/* The three 50-bin data histograms in the order Close, Separated, DecayTag
 * (FakeLikelihood.H:24-26, bins 1..50) and Corrections.ExposureRatio (:107). */
int smcmc_fake_set_data(smcmc_engine* e, const double* data150, double exposure);
/* FakeLikelihood::FillHistograms (:188-216) at m points: out[m*150] simulated
 * bin contents, same order as data150. */
int smcmc_fake_histograms(smcmc_engine* e, const double* x, int m, double* out);
/* The exact integer event counts behind those histograms, per weight class:
 * out[m*450], slot layout of DESIGN.md section 3 (signal/background x decay tag
 * x histogram x bin).  Test and diagnostics access. */
int smcmc_fake_counts(smcmc_engine* e, const double* x, int m, uint32_t* out);
/* Diagnostic for the pair kernel's FP32 interval filter (DESIGN.md section 3):
 * evaluates EVERY (point, event) pair both ways and returns out3 = {pairs,
 * pairs the filter left to FP64, pairs where a filter decision differs from
 * the FP64 decision}.  The last number must be 0. */
int smcmc_fake_filter_check(smcmc_engine* e, const double* x, int m, uint64_t* out3);
/* Diagnostic for the pair kernel's tile skip (DESIGN.md section 4.1): for each
 * warp of 32 consecutive points and each event tile of the candidate mass bands,
 * applies the kernel's skip rule, and checks every pair of every skipped tile in
 * FP64.  out3 = {tiles tested, tiles skipped, pairs of skipped tiles that the
 * FP64 arithmetic counts}.  The last number must be 0. */
int smcmc_fake_skip_check(smcmc_engine* e, const double* x, int m, uint64_t* out3);
/* SMCMC_LLH_UNBINNED, the unbinned counterpart of the event likelihood.  The
 * reference has no such functor (its likelihood is binned); this one is DEFINED
 * HERE on top of the reference's per-event corrections, with the same 9
 * parameters (example/SystematicCorrection.H:11-22):
 *   L(p) = sum over events of log( w_s phi_s(m') + w_b phi_b(m') )
 *   log m' = corrected log-mass of InvariantMass (:50-79)
 *   w_s, w_b = EventWeight (:81-117) of the signal / background hypothesis for
 *              the event's MuDk flag (exposure ratio 1); the event's Type is not used
 *   phi_s(m) = log-normal density, mean of log m = log 135, sigma = log 1.3
 *   phi_b(m) = exp(-m/500)/500
 * Its CPU checker is oracle/smcmc_oracle.cc (EvalUnbinned); parity is not pinned by
 * the reference.  Events are copied to the device and kept in upload order inside
 * the two MuDk classes. */
int smcmc_unbinned_set_events(smcmc_engine* e, const smcmc_event* events, int64_t n);
/* TDummyLogLikelihood::Error (TDummyLogLikelihood.H:147), n x n row-major. */
int smcmc_dummy_set_error(smcmc_engine* e, const double* error, int n);
/* How the dense contractions of TDummyLogLikelihood (likelihood :21-31, gradient
 * :34-42) are evaluated.  EXACT (default): the reference's operation order,
 * multiply and add rounded separately -- bit-identical to the host functor.
 * TENSOR: X . Error^T on the FP64 tensor cores (DMMA), fused multiply-adds in the
 * tensor core's summation order -- within 1e-12 relative, not bit for bit; meant
 * for dimensions of a few hundred and thousands of chains. */
typedef enum smcmc_dummy_mode { SMCMC_DUMMY_EXACT = 0, SMCMC_DUMMY_TENSOR = 1 } smcmc_dummy_mode;
int smcmc_dummy_set_mode(smcmc_engine* e, int mode);

/* ---- sampler ------------------------------------------------------------- */
/* UserLikelihood::operator() at m arbitrary points (x[m*dim]) -> llh[m]. */
int smcmc_eval(smcmc_engine* e, const double* x, int m, double* llh);
/* TSimpleMCMC::Start (:246-276): x0[chains*dim]; ok[chains] (may be NULL)
 * receives the per-chain return value. */
int smcmc_start(smcmc_engine* e, const double* x0, int32_t* ok);
/* nsteps calls of TSimpleMCMC::Step(false, metropolis) (:370-496) on every
 * chain.  Asynchronous: returns after queueing the launches. */
int smcmc_step(smcmc_engine* e, int nsteps, int metropolis);
/* nsteps calls of Step(true, metropolis): as smcmc_step, then copies the
 * per-step quantities a TTree::Fill would have recorded to host memory.
 * Synchronous. */
int smcmc_step_trace(smcmc_engine* e, int nsteps, int metropolis,
                     const smcmc_trace* trace);
/* Read a per-chain quantity (synchronous). */
int smcmc_get(smcmc_engine* e, int field, void* dst, size_t bytes);

/* ---- checkpoint / resume ----------------------------------------------------- */
/* What the reference keeps in its output tree to continue a chain
 * (TSimpleMCMC.H:208-216 and the Adaptive* branches :1616-1626, filled by
 * SaveStep(true) :528-532,1631-1652), for every chain of the engine.  Arrays
 * are chain-major; covariance packed lower-triangular as the
 * AdaptiveCovariance branch. */
typedef struct smcmc_saved_state {
    double* accepted;            /* [chains*dim]  Accepted                    */
    double* log_likelihood;      /* [chains]      LogLikelihood               */
    int32_t* total_steps;        /* [chains]      TotalSteps                  */
    double* step_rms;            /* [chains]      StepRMS                     */
    int32_t* trials;             /* [chains]      AdaptiveTrials              */
    int32_t* successes;          /* [chains]      AdaptiveSuccesses           */
    int32_t* next_update;        /* [chains]      AdaptiveNextUpdate          */
    double* acceptance;          /* [chains]      AdaptiveAcceptance          */
    double* acceptance_trials;   /* [chains]      AdaptiveAcceptanceTrials    */
    double* sigma;               /* [chains]      AdaptiveSigma               */
    double* central_point;       /* [chains*dim]  AdaptiveCentralPoint        */
    double* central_point_trials;/* [chains]      AdaptiveCentralPointTrials  */
    double* covariance;          /* [chains*dim*(dim+1)/2] AdaptiveCovariance */
    double* covariance_trials;   /* [chains]      AdaptiveCovarianceTrials    */
    double* covariance_trace;    /* [chains]      AdaptiveCovarianceTrace (GetCovarianceTrace :961-967);
                                    written by smcmc_save_state, not read by smcmc_restore_state */
} smcmc_saved_state;
/* SaveStep(true): copy the state of every chain into the caller's arrays. */
int smcmc_save_state(smcmc_engine* e, const smcmc_saved_state* out);
/* TSimpleMCMC::Restore (:282-352) + TProposeAdaptiveStep::RestoreState
 * (:1501-1610) on every chain, after Start(): adopt the saved point and
 * proposal state, re-evaluate the likelihood at the restored point (the
 * calculated value replaces the saved one when they differ by more than 1e-4,
 * :335-345; mismatch[c] receives 1 in that case, may be NULL), set the sigma
 * trace to the trace of the restored covariance and run UpdateProposal(). */
int smcmc_restore_state(smcmc_engine* e, const smcmc_saved_state* in, int32_t* mismatch);
/* The step counter that addresses the random stream: a resumed run continues
 * the stream where the saved run stopped when this is carried over. */
int smcmc_get_step_index(smcmc_engine* e, uint32_t* step);
int smcmc_set_step_index(smcmc_engine* e, uint32_t step);

/* ---- Hamiltonian Monte Carlo: sMCMC::TSimpleHMC<L, G> (TSimpleHMC.H:119-973) ---- */
/* The same engine handle (likelihood, dim, chains, seed, likelihood inputs) can
 * be driven as an ensemble of TSimpleHMC chains instead of TSimpleMCMC chains.
 * Random draws of chain c at step s: slots 0..dim-1 the momentum refresh (:568,
 * only when alpha < 1), the next slot the step-size jitter (:297), the next one
 * the accept test (:347). */
typedef enum smcmc_hmc_setting {
    SMCMC_HMC_ALPHA = 0,            /* SetAlpha        :175                                  */
    SMCMC_HMC_MEAN_EPSILON = 1,     /* SetMeanEpsilon  :181 (Start() resets it to 0.05, :229) */
    SMCMC_HMC_LEAPFROG = 2,         /* SetLeapFrog     :190 (stored negated = fixed)          */
    SMCMC_HMC_USER_GRADIENT = 3,    /* 1: TSimpleHMC<L, L> (the likelihood's own gradient functor,
                                       TDummyLogLikelihood.H:34-42, THardLogLikelihood.H:72-91, or
                                       smcmc_user_ops::gradient); 0: TSimpleHMC<L>, finite
                                       differences (:417-444).  Set before smcmc_hmc_start.   */
    SMCMC_HMC_KEEP_ERROR_MATRIX = 4,/* 1: keep fEstimatedError per chain (dim*dim doubles), which
                                       gradient type 2 (:447-454) reads.  Set before start.   */
    SMCMC_HMC_POOLED_COVARIANCE = 5 /* NEW (not in the reference): UpdateCovariance / UpdateErrorMatrix
                                       (:665-858) on ONE estimate pooled over every chain of the engine
                                       instead of one per chain -- the estimate only feeds the step-size
                                       and trajectory-length tuning (:833-847) unless gradient type 2 is
                                       used.  0 per chain (the reference), 1 pooled, -1 (default) pooled
                                       when the per-chain triangles would take >= 256 MB.  Before start. */
} smcmc_hmc_setting;

/* Per-chain quantities readable with smcmc_hmc_get(); arrays chain-major. */
typedef enum smcmc_hmc_field {
    SMCMC_HMC_F_ACCEPTED = 0,      /* double[chains*dim]      fAccepted                      */
    SMCMC_HMC_F_MOMENTUM = 1,      /* double[chains*dim]      fAcceptedMomentum              */
    SMCMC_HMC_F_PROPOSED = 2,      /* double[chains*dim]      fProposed                      */
    SMCMC_HMC_F_CENTRAL = 3,       /* double[chains*dim]      GetCentralPoint        :193    */
    SMCMC_HMC_F_AVERAGE = 4,       /* double[chains*dim]      fAveragePoint                  */
    SMCMC_HMC_F_COVARIANCE = 5,    /* double[chains*dim*dim]  GetEstimatedCovariance :197    */
    SMCMC_HMC_F_ERROR_MATRIX = 6,  /* double[chains*dim*dim]  fEstimatedError                */
    SMCMC_HMC_F_SCALARS = 7,       /* double[chains*SMCMC_HMC_SCALAR_COUNT], columns below   */
    /* pooled covariance (SMCMC_HMC_POOLED_COVARIANCE) */
    SMCMC_HMC_F_POOLED_COVARIANCE = 8, /* double[dim*dim]  the ensemble's fEstimatedCovariance      */
    SMCMC_HMC_F_POOLED_AVERAGE = 9,    /* double[dim]      the ensemble's fAveragePoint             */
    SMCMC_HMC_F_POOLED_SCALARS = 10    /* double[SMCMC_HMC_POOLED_SCALAR_COUNT], columns below      */
} smcmc_hmc_field;
enum {
    SMCMC_HMC_PS_TRIALS = 0,         /* samples (chain-steps) behind the estimate                */
    SMCMC_HMC_PS_EST_COV_TRACE,      /* fEstimatedCovarianceTrace                                */
    SMCMC_HMC_PS_CUR_COV_TRACE,      /* fCurrentCovarianceTrace                                  */
    SMCMC_HMC_PS_ORBIT_LENGTH,       /* fEstimatedOrbitLength                                    */
    SMCMC_HMC_PS_MAX_SCALE,          /* sqrt(largest |eigenvalue|), clamped (:820-825)           */
    SMCMC_HMC_PS_MIN_SCALE,          /* sqrt(smallest |eigenvalue|), clamped                     */
    SMCMC_HMC_PS_STEP_COUNT,         /* steps that contributed                                   */
    SMCMC_HMC_PS_UPDATES,            /* UpdateErrorMatrix bodies run so far                      */
    SMCMC_HMC_PS_REPAIRED,           /* the last update found the estimate not positive definite */
    SMCMC_HMC_POOLED_SCALAR_COUNT
};
enum {
    SMCMC_HMC_S_ACCEPTANCE = 0,      /* GetAcceptanceRate :160 */
    SMCMC_HMC_S_MEAN_EPSILON,        /* GetMeanEpsilon    :184 */
    SMCMC_HMC_S_LEAPFROG,            /* fLeapFrogSteps         */
    SMCMC_HMC_S_REVERSAL_LEN,
    SMCMC_HMC_S_ACCEPTED_POTENTIAL,
    SMCMC_HMC_S_PROPOSED_POTENTIAL,
    SMCMC_HMC_S_CENTRAL_POTENTIAL,   /* GetCentralPotential :194 */
    SMCMC_HMC_S_POTENTIAL_COUNT,     /* GetPotentialCount :163 */
    SMCMC_HMC_S_GRADIENT_COUNT,      /* GetGradientCount  :168 */
    SMCMC_HMC_S_STEP_COUNT,
    SMCMC_HMC_S_COV_TRIALS,
    SMCMC_HMC_S_AVERAGE_TRIALS,
    SMCMC_HMC_S_EST_COV_TRACE,
    SMCMC_HMC_S_CUR_COV_TRACE,
    SMCMC_HMC_S_ORBIT_LENGTH,
    SMCMC_HMC_S_STEPS_REMAINING,
    SMCMC_HMC_S_STEPS_SINCE_UPDATE,
    SMCMC_HMC_SCALAR_COUNT
};

/* Optional per-step record of smcmc_hmc_step_trace(): what SaveStep() (:861)
 * writes to the tree (:139-147).  Step-major, any pointer may be NULL. */
typedef struct smcmc_hmc_trace {
    double* potential;      /* [nsteps*chains]      "LogLikelihood" = fAcceptedPotential */
    double* points;         /* [nsteps*chains*dim]  "Accepted"                           */
    double* mean_epsilon;   /* [nsteps*chains]      "MeanEpsilon"                        */
    int32_t* leapfrog;      /* [nsteps*chains]      "Leapfrog"                           */
    int32_t* accepted;      /* [nsteps*chains]      1 when the proposed point was taken  */
} smcmc_hmc_trace;

int smcmc_hmc_set(smcmc_engine* e, int setting, double value);
/* TSimpleHMC::Start (:210-269): x0[chains*dim]. */
int smcmc_hmc_start(smcmc_engine* e, const double* x0);
/* TSimpleHMC::SetPosition (:202-205): x[chains*dim]. */
int smcmc_hmc_set_position(smcmc_engine* e, const double* x);
/* nsteps calls of TSimpleHMC::Step(false, gradient_type) (:279-401) on every
 * chain.  gradient_type as PotentialGradient (:467-532): 0/1 user gradient when
 * there is one, else finite differences; 2 covariant; 3 finite differences;
 * 4 user gradient or SMCMC_ERR_LOGIC; 5 zero. */
int smcmc_hmc_step(smcmc_engine* e, int nsteps, int gradient_type);
int smcmc_hmc_step_trace(smcmc_engine* e, int nsteps, int gradient_type, const smcmc_hmc_trace* trace);
int smcmc_hmc_get(smcmc_engine* e, int field, void* dst, size_t bytes);

/* ---- instrumentation ------------------------------------------------------ */
/* Kernel launches issued by this engine so far. */
int64_t smcmc_launch_count(const smcmc_engine* e);
/* Device time (ms, CUDA events on the engine's stream) and launch count
 * accumulated by the dominant event-pair kernel since the last reset. */
int smcmc_pair_kernel_stats(smcmc_engine* e, double* total_ms, int64_t* launches,
                            int reset);
/* Enable (1) / disable (0) CUDA-event timing of the dominant kernel. */
int smcmc_enable_kernel_timing(smcmc_engine* e, int on);

/* Measured FP64 FMA throughput of `device` in TFLOP/s (2 flop per DFMA): a
 * register-resident chain of independent DFMAs on every SM, timed with CUDA
 * events.  The roofline denominator for the FP64-bound pair kernel. */
int smcmc_measure_fp64_peak(int device, double* tflops);
/* Measured throughput of the FP64 tensor cores of `device` in TFLOP/s: register-resident
 * chains of independent mma.sync.m8n8k4.f64 (DMMA, 512 flop per warp instruction) on every
 * SM.  The roofline denominator of the dense contractions (kDummyContractDmma,
 * kPoolAccumulateDmma). */
int smcmc_measure_dmma_peak(int device, double* tflops);
/* Measured throughput of the special-function unit of `device` in 10^9 ex2
 * evaluations per second (register-resident chains of independent MUFU.EX2 on
 * every SM).  The roofline denominator of the event-pair kernel, which needs two
 * exponentials per (chain, event) pair. */
int smcmc_measure_sfu_peak(int device, double* gops);
/* ---- ensemble diagnostics (SURVEY.md 8f rank 3) ------------------------------
 * The reference derives these offline from the output TTree, one chain at a
 * time: MakeCovariance.C:63-89 (mean and covariance of the accepted points),
 * MakeAutocorrelation.C:96-148 (autocorrelation on a subset of lags).  Here the
 * sums are accumulated on the device for every chain after every smcmc_step,
 * so the points of a large ensemble never have to be written out.  R-hat is
 * Gelman-Rubin's potential scale reduction across the chains of the engine. */
typedef struct smcmc_diag_result {
    int64_t* samples;         /* [1] chains x steps accumulated                                  */
    int64_t* steps;           /* [1] steps accumulated                                           */
    double* mean;             /* [n]   sum x / N                         MakeCovariance.C:76     */
    double* covariance;       /* [n*n] sum x_i x_j / N - mean_i mean_j   MakeCovariance.C:79-83  */
    double* rhat;             /* [n]   sqrt(((N-1)/N W + B/N) / W) over the chains               */
    int32_t* lags;            /* [nlags] the sampled lags 1,2,3,4,6,8,12,... <= max_lag          */
    double* autocorrelation;  /* [nlags*n] (<x(t) x(t-lag)> - mean^2) / var, lag-major
                                                                     MakeAutocorrelation.C:131-136 */
    double* tau;              /* [n] integrated autocorrelation time 1 + 2 sum rho(k)             */
    double* ess;              /* [n] samples / tau                                                */
} smcmc_diag_result;          /* any pointer may be NULL                                          */
/* Start accumulating (MH engines, smcmc_step / smcmc_step_trace).  max_lag = 0:
 * no autocorrelation; otherwise a ring buffer of max_lag points per chain is kept
 * on the device (max_lag x chains x dim doubles). */
int smcmc_diag_enable(smcmc_engine* e, int max_lag);
int smcmc_diag_reset(smcmc_engine* e);
int smcmc_diag_lag_count(smcmc_engine* e, int32_t* nlags);
int smcmc_diag_get(smcmc_engine* e, const smcmc_diag_result* out);

/* Device self-test of the shared-divisor division of the staged covariance
 * update (csrc/proposal_staged.cuh, replacing the per-entry division of
 * TSimpleMCMC.H:1811): `count` random numerators and divisors are divided both
 * ways; *mismatches receives the number of quotients that differ in any bit
 * from the correctly rounded IEEE quotient. */
int smcmc_selftest_division(int device, int64_t count, uint64_t seed, int64_t* mismatches);

#ifdef __cplusplus
}
#endif
#endif
