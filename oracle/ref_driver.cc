// oracle/ref_driver.cc -- builds oracle/_ref/libsmcmc_ref.so.
//
// This translation unit #includes the reference's OWN headers, unmodified,
// from a checkout of the reference project (never copied into this repo)
// and exposes them through the single-chain C interface of chain_api.h.
// ROOT is replaced by oracle/rootshim.  The reference's global gRandom is
// pointed at an injected generator that serves the counter-based stream of
// include/smcmc_rng.h, so the reference consumes exactly the draws the device
// consumes.  TEST INFRASTRUCTURE ONLY (see chain_api.h).
//
// Build: oracle/Makefile target `ref` (needs REFERENCE=<reference checkout>).

// Standard and shim headers first, so that the access-specifier override
// below only touches the reference's own classes.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <iomanip>
#include <iostream>
#include <limits>
#include <sstream>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <vector>

#include <TDecompChol.h>
#include <TFile.h>
#include <TH1D.h>
#include <TMatrixD.h>
#include <TMatrixDSymEigen.h>
#include <TRandom.h>
#include <TRandom3.h>
#include <TTree.h>
#include <TVectorD.h>

#include "chain_api.h"
#include "smcmc_rng.h"

// Read-only test access to the proposal's covariance and decomposition.
#define private public
#define protected public
#include "TSimpleMCMC.H"
using namespace sMCMC;  // example/ predates the namespace (SURVEY.md F7)
#include "TProposeVAATStep.H"
#include "TDummyLogLikelihood.H"
#include "THorrificLogLikelihood.H"
#include "TAsymLogLikelihood.H"
// THorrificLogLikelihood.H reuses the include guard of THardLogLikelihood.H
// (a copy-paste quirk of the reference): release it so that both can be used.
#undef THardLogLikelihood_H_seen
#include "THardLogLikelihood.H"
#include "example/FakeLikelihood.H"
#include "example4/TConstrainedLikelihood.H"
#define HMC_DEBUG_LEVEL -1
#include "TSimpleHMC.H"
#undef private
#undef protected

// oracle/ref_ex2.cc: the reference's example2 likelihood (own translation unit)
extern "C" {
void* ref_ex2_create(void);
void ref_ex2_destroy(void* h);
int ref_ex2_set(void* h, const orc_event* ev, long n, const double* data150);
double ref_ex2_llh(void* h, const double* x, int n);
int ref_ex2_hist(void* h, const double* x, int n, double* out150);
}

namespace {

std::string gLastError;

// example2's FakeLikelihood behind the likelihood-functor contract
// (TSimpleMCMC.H:59-106): TSimpleMCMC holds it by value and calls operator().
class Example2Likelihood {
public:
    Example2Likelihood() : impl(ref_ex2_create()) {}
    ~Example2Likelihood() { ref_ex2_destroy(impl); }
    Example2Likelihood(const Example2Likelihood&) = delete;
    double operator()(const Vector& point) { return ref_ex2_llh(impl, point.data(), (int)point.size()); }
    void* impl;
};

// gRandom replacement: call k of step s of chain c returns slot k.
class InjectedRandom : public TRandom {
public:
    InjectedRandom(uint64_t seed, uint32_t chain)
        : fSeed(seed), fChain(chain), fStep(0), fSlot(0) {}
    void Begin(uint32_t step) { fStep = step; fSlot = 0; }
    virtual double Rndm() {
        return smcmc_uniform(fSeed, fChain, fStep, fSlot++, SMCMC_STREAM_STEP);
    }
    virtual double UnitGaus() {
        return smcmc_normal(fSeed, fChain, fStep, fSlot++, SMCMC_STREAM_STEP);
    }
private:
    uint64_t fSeed;
    uint32_t fChain, fStep, fSlot;
};

// The documentation example likelihood, TSimpleMCMC.H:111-120.
class UnitGaussLikelihood {
public:
    double operator()(const Vector& point) const {
        double logLikelihood = 0.0;
        for (std::size_t i = 0; i < point.size(); ++i) {
            logLikelihood += -0.5 * point[i] * point[i];
        }
        return logLikelihood;
    }
};

struct ChainBase {
    InjectedRandom rng;
    uint32_t step;
    int dim;
    ChainBase(uint64_t seed, uint32_t chain, int d)
        : rng(seed, chain), step(0), dim(d) {}
    virtual ~ChainBase() {}
    virtual TProposeAdaptiveStep& Prop() = 0;
    virtual bool Start(const Vector& x) = 0;
    virtual bool Step(int metropolis) = 0;
    virtual bool StepSaved(int metropolis) = 0;
    virtual double Llh(const Vector& x) = 0;
    virtual const Vector& Accepted() = 0;
    virtual double AcceptedLlh() = 0;
    virtual double ProposedLlh() = 0;
    virtual double StepRMS() = 0;
    virtual int TotalSteps() = 0;
    virtual int LlhCalls() = 0;
    virtual void SetStepRMSWindow(int n) = 0;
    virtual void SaveStep() = 0;
    virtual void Restore(TTree* tree) = 0;
    virtual void RestoreRandom(TTree* tree) = 0;
    virtual FakeLikelihood* Fake() { return 0; }
    virtual void* Fake2() { return 0; }
    virtual TProposeVAATStep* Vaat() { return 0; }
    TTree tree;      // every chain writes to its own in-memory tree
};

template <class L, class P = TProposeAdaptiveStep>
struct Chain : public ChainBase {
    static const bool kAdaptive = std::is_same<P, TProposeAdaptiveStep>::value;
    TSimpleMCMC<L, P> mcmc;
    Chain(uint64_t seed, uint32_t chain, int d)
        : ChainBase(seed, chain, d), mcmc(&tree, false) {}
    void SaveStep() { mcmc.SaveStep(); }
    // TProposeVAATStep::RestoreState does not match the call in
    // TSimpleMCMC::Restore (TProposeVAATStep.H:33 vs TSimpleMCMC.H:351): Restore
    // can only be instantiated for the adaptive proposal.
    void Restore(TTree* t) {
        if constexpr (kAdaptive) mcmc.Restore(t);
        else throw std::logic_error("Restore needs TProposeAdaptiveStep");
    }
    void RestoreRandom(TTree* t) {
        if constexpr (kAdaptive) mcmc.Restore(t, true);
        else throw std::logic_error("Restore needs TProposeAdaptiveStep");
    }
    bool StepSaved(int metropolis) { return mcmc.Step(true, metropolis); }
    TProposeAdaptiveStep& Prop() {
        if constexpr (kAdaptive) return mcmc.GetProposeStep();
        else throw std::logic_error("not a TProposeAdaptiveStep chain");
    }
    TProposeVAATStep* Vaat() {
        if constexpr (kAdaptive) return 0;
        else return &mcmc.GetProposeStep();
    }
    bool Start(const Vector& x) { return mcmc.Start(x, false); }
    bool Step(int metropolis) { return mcmc.Step(false, metropolis); }
    double Llh(const Vector& x) { return mcmc.GetLogLikelihood()(x); }
    const Vector& Accepted() { return mcmc.GetAccepted(); }
    double AcceptedLlh() { return mcmc.GetAcceptedLogLikelihood(); }
    double ProposedLlh() { return mcmc.GetProposedLogLikelihood(); }
    double StepRMS() { return mcmc.GetStepRMS(); }
    int TotalSteps() { return mcmc.fTotalSteps; }
    int LlhCalls() { return mcmc.GetLogLikelihoodCount(); }
    void SetStepRMSWindow(int n) { mcmc.SetStepRMSWindow(n); }
};

struct FakeChain : public Chain<FakeLikelihood> {
    FakeChain(uint64_t seed, uint32_t chain, int d)
        : Chain<FakeLikelihood>(seed, chain, d) {
        FakeLikelihood& like = mcmc.GetLogLikelihood();
        like.DataClose = like.DataSeparated = like.DataDecayTag = 0;
        like.SimulatedClose = like.SimulatedSeparated = like.SimulatedDecayTag = 0;
    }
    FakeLikelihood* Fake() { return &mcmc.GetLogLikelihood(); }
};

struct FakeVaatChain : public Chain<FakeLikelihood, TProposeVAATStep> {
    FakeVaatChain(uint64_t seed, uint32_t chain, int d)
        : Chain<FakeLikelihood, TProposeVAATStep>(seed, chain, d) {
        FakeLikelihood& like = mcmc.GetLogLikelihood();
        like.DataClose = like.DataSeparated = like.DataDecayTag = 0;
        like.SimulatedClose = like.SimulatedSeparated = like.SimulatedDecayTag = 0;
    }
    FakeLikelihood* Fake() { return &mcmc.GetLogLikelihood(); }
};

struct Fake2Chain : public Chain<Example2Likelihood> {
    Fake2Chain(uint64_t seed, uint32_t chain, int d) : Chain<Example2Likelihood>(seed, chain, d) {}
    void* Fake2() { return mcmc.GetLogLikelihood().impl; }
};

ChainBase* H(void* h) { return static_cast<ChainBase*>(h); }

template <class F>
int Guard(F f) {
    try {
        return f();
    } catch (std::exception& e) {
        gLastError = e.what();
        return -1;
    }
}

}  // namespace

extern "C" {

const char* ref_last_error(void) { return gLastError.c_str(); }

void* ref_chain_create(int kind, int dim, uint64_t seed, uint32_t chain) {
    ChainBase* c = 0;
    switch (kind) {
    case ORC_LLH_UNIT_GAUSS:
        c = new Chain<UnitGaussLikelihood>(seed, chain, dim);
        break;
    case ORC_LLH_DUMMY: {
        // As shipped: dim 100, VERY_CORRELATED (TDummyLogLikelihood.H:16,78).
        Chain<TDummyLogLikelihood>* d = new Chain<TDummyLogLikelihood>(seed, chain, 100);
        if (dim != 100) { delete d; gLastError = "reference TDummyLogLikelihood is 100-dim"; return 0; }
        std::streambuf* old = std::cout.rdbuf(0);
        d->mcmc.GetLogLikelihood().Init();
        std::cout.rdbuf(old);
        c = d;
        break;
    }
    case ORC_LLH_HORRIFIC:
        if (dim != 75) { gLastError = "reference THorrificLogLikelihood is 75-dim"; return 0; }
        c = new Chain<THorrificLogLikelihood>(seed, chain, 75);
        break;
    case ORC_LLH_ASYM:
        if (dim != 100) { gLastError = "reference TASymLogLikelihood is 100-dim"; return 0; }
        c = new Chain<TASymLogLikelihood>(seed, chain, 100);
        break;
    case ORC_LLH_HARD:
        if (dim != 6) { gLastError = "reference THardLogLikelihood is 6-dim"; return 0; }
        c = new Chain<THardLogLikelihood>(seed, chain, 6);
        break;
    case ORC_LLH_FAKE:
        if (dim != (int)SystematicCorrection::kParamSize) { gLastError = "FakeLikelihood is 9-dim"; return 0; }
        c = new FakeChain(seed, chain, dim);
        break;
    case ORC_LLH_FAKE2:
        if (dim != 9) { gLastError = "example2 FakeLikelihood is 9-dim"; return 0; }
        c = new Fake2Chain(seed, chain, dim);
        break;
    case ORC_LLH_CONSTRAINED: {
        Chain<TConstrainedLikelihood>* k = new Chain<TConstrainedLikelihood>(seed, chain, 25);
        k->mcmc.GetLogLikelihood().Init();                       // example4/Constrained.C:21-22
        if (dim != (int)k->mcmc.GetLogLikelihood().GetDim()) { delete k; gLastError = "TConstrainedLikelihood is 25-dim"; return 0; }
        c = k;
        break;
    }
    default:
        gLastError = "unknown likelihood kind";
        return 0;
    }
    c->Prop().SetDim(c->dim);
    return c;
}

// TSimpleMCMC<L, TProposeVAATStep>, the pairing of SimpleVAAT.C:31.
void* ref_chain_create_vaat(int kind, int dim, uint64_t seed, uint32_t chain) {
    ChainBase* c = 0;
    switch (kind) {
    case ORC_LLH_UNIT_GAUSS:
        c = new Chain<UnitGaussLikelihood, TProposeVAATStep>(seed, chain, dim);
        break;
    case ORC_LLH_HORRIFIC:
        if (dim != 75) { gLastError = "reference THorrificLogLikelihood is 75-dim"; return 0; }
        c = new Chain<THorrificLogLikelihood, TProposeVAATStep>(seed, chain, 75);
        break;
    case ORC_LLH_ASYM:
        if (dim != 100) { gLastError = "reference TASymLogLikelihood is 100-dim"; return 0; }
        c = new Chain<TASymLogLikelihood, TProposeVAATStep>(seed, chain, 100);
        break;
    case ORC_LLH_FAKE:
        if (dim != 9) { gLastError = "FakeLikelihood is 9-dim"; return 0; }
        c = new FakeVaatChain(seed, chain, dim);
        break;
    default:
        gLastError = "likelihood kind not offered with TProposeVAATStep";
        return 0;
    }
    c->Vaat()->SetDim(c->dim);
    return c;
}

int ref_chain_get_vaat(void* h, double* sigma, double* acceptance, int32_t* acceptanceTrials, int32_t* misc) {
    TProposeVAATStep* p = H(h)->Vaat();
    if (!p) { gLastError = "not a TProposeVAATStep chain"; return -1; }
    if (sigma) std::copy(p->fSigma.begin(), p->fSigma.end(), sigma);
    if (acceptance) std::copy(p->fAcceptance.begin(), p->fAcceptance.end(), acceptance);
    if (acceptanceTrials) std::copy(p->fAcceptanceTrials.begin(), p->fAcceptanceTrials.end(), acceptanceTrials);
    if (misc) {
        misc[0] = p->GetTrials();
        misc[1] = p->GetSuccesses();
        misc[2] = p->fLastIndex;
        misc[3] = (int32_t)p->fNextIndex.size();
    }
    return 0;
}

void ref_chain_destroy(void* h) { delete H(h); }

int ref_chain_set_fake(void* h, const orc_event* ev, long n,
                       const double* data150, double exposure) {
    if (H(h)->Fake2()) return ref_ex2_set(H(h)->Fake2(), ev, n, data150);
    FakeLikelihood* like = H(h)->Fake();
    if (!like) { gLastError = "not a FakeLikelihood chain"; return -1; }
    static_assert(sizeof(Simulated::Event) == sizeof(orc_event), "event layout");
    like->SimulatedSample.resize(n);
    std::memcpy((void*)like->SimulatedSample.data(), ev, sizeof(orc_event) * n);
    // Same histogram geometry as FakeData::FillData (example/FakeData.H:94-104).
    TH1D* close = new TH1D("DataClose", "", 50, 0.0, 500.0);
    TH1D* separated = new TH1D("DataSeparated", "", 50, 0.0, 500.0);
    TH1D* tag = new TH1D("DataDecayTag", "", 50, 0.0, 500.0);
    for (int b = 0; b < 50; ++b) {
        close->SetBinContent(b + 1, data150[b]);
        separated->SetBinContent(b + 1, data150[50 + b]);
        tag->SetBinContent(b + 1, data150[100 + b]);
    }
    like->DataClose = close;
    like->DataSeparated = separated;
    like->DataDecayTag = tag;
    like->SimulatedSeparated = (TH1D*)separated->Clone("simSeparated");
    like->SimulatedClose = (TH1D*)close->Clone("simClose");
    like->SimulatedDecayTag = (TH1D*)tag->Clone("simDecayTag");
    like->Corrections.ExposureRatio = exposure;
    return 0;
}

int ref_chain_set_error_matrix(void*, const double*, int) {
    gLastError = "the reference builds its own error matrix in Init()";
    return -1;
}

int ref_chain_set(void* h, int field, double v) {
    if (H(h)->Vaat() && field != ORC_SET_STEP_RMS_WINDOW) {
        if (field == ORC_SET_ACCEPTANCE_WINDOW) H(h)->Vaat()->SetAcceptanceWindow(v);
        else if (field == ORC_SET_ACCEPTANCE_RIGIDITY) H(h)->Vaat()->SetAcceptanceRigidity(v);
        else { gLastError = "TProposeVAATStep has no such setting"; return -1; }
        return 0;
    }
    if (H(h)->Vaat()) { H(h)->SetStepRMSWindow((int)v); return 0; }
    TProposeAdaptiveStep& p = H(h)->Prop();
    switch (field) {
    case ORC_SET_SIGMA: p.SetSigma(v); break;
    case ORC_SET_TARGET_ACCEPTANCE: p.SetTargetAcceptance(v); break;
    case ORC_SET_ACCEPTANCE_WINDOW: p.SetAcceptanceWindow(v); break;
    case ORC_SET_ACCEPTANCE_RIGIDITY: p.SetAcceptanceRigidity(v); break;
    case ORC_SET_ACCEPTANCE_DEWEIGHT: p.SetAcceptanceUpdateDeweighting(v); break;
    case ORC_SET_COVARIANCE_WINDOW: p.SetCovarianceWindow((int)v); break;
    case ORC_SET_COVARIANCE_DEWEIGHT: p.SetCovarianceUpdateDeweighting(v); break;
    case ORC_SET_COVARIANCE_FROZEN: p.SetCovarianceFrozen(v != 0.0); break;
    case ORC_SET_COVARIANCE_TRIALS: p.SetCovarianceTrials(v); break;
    case ORC_SET_CENTER_TRIALS: p.SetEstimatedCenterTrials(v); break;
    case ORC_SET_NEXT_UPDATE: p.SetNextUpdate(v); break;
    case ORC_SET_MAX_CORRELATION: p.SetMaximumCorrelation(v); break;
    case ORC_SET_STEP_RMS_WINDOW: H(h)->SetStepRMSWindow((int)v); break;
    default: gLastError = "unknown field"; return -1;
    }
    return 0;
}

int ref_chain_set_gaussian(void* h, int d, double sigma) {
    if (H(h)->Vaat()) { H(h)->Vaat()->SetGaussian(d, sigma); return 0; }
    H(h)->Prop().SetGaussian(d, sigma);
    return 0;
}

int ref_chain_set_uniform(void* h, int d, double lo, double hi) {
    if (H(h)->Vaat()) { H(h)->Vaat()->SetUniform(d, lo, hi); return 0; }
    H(h)->Prop().SetUniform(d, lo, hi);
    return 0;
}

int ref_chain_set_correlation(void* h, int d1, int d2, double c) {
    H(h)->Prop().SetCorrelation(d1, d2, c);
    return 0;
}

int ref_chain_start(void* h, const double* x0) {
    ChainBase* c = H(h);
    return Guard([&]() {
        gRandom = &c->rng;
        Vector x(x0, x0 + c->dim);
        return c->Start(x) ? 1 : 0;
    });
}

int ref_chain_step(void* h, int nsteps, int metropolis, int32_t* accepted,
                   double* llhAccepted, double* llhProposed, double* x,
                   double* sigma) {
    ChainBase* c = H(h);
    return Guard([&]() {
        gRandom = &c->rng;
        for (int s = 0; s < nsteps; ++s) {
            c->rng.Begin(c->step++);
            bool ok = c->Step(metropolis);
            if (accepted) accepted[s] = ok ? 1 : 0;
            if (llhAccepted) llhAccepted[s] = c->AcceptedLlh();
            if (llhProposed) llhProposed[s] = c->ProposedLlh();
            if (sigma) sigma[s] = c->Vaat() ? c->Vaat()->GetSigma() : c->Prop().GetSigma();
            if (x) std::copy(c->Accepted().begin(), c->Accepted().end(),
                             x + (size_t)s * c->dim);
        }
        return 0;
    });
}

// Step(true): as ref_chain_step but every step is written to the chain's tree.
int ref_chain_step_saved(void* h, int nsteps, int32_t* accepted) {
    ChainBase* c = H(h);
    return Guard([&]() {
        gRandom = &c->rng;
        for (int s = 0; s < nsteps; ++s) {
            c->rng.Begin(c->step++);
            bool ok = c->StepSaved(0);
            if (accepted) accepted[s] = ok ? 1 : 0;
        }
        return 0;
    });
}

// SaveStep(): the full proposal state goes to the tree (TSimpleMCMC.H:528-532).
int ref_chain_save_step(void* h) {
    return Guard([&]() { H(h)->SaveStep(); return 0; });
}

// Restore(tree) from the tree of another chain (TSimpleMCMC.H:282-352); the
// random stream continues at the source chain's step counter.
int ref_chain_restore(void* h, void* source) {
    ChainBase* c = H(h);
    ChainBase* src = H(source);
    return Guard([&]() {
        gRandom = &c->rng;
        c->Restore(&src->tree);
        c->step = src->step;
        return 0;
    });
}

int ref_chain_restore_random(void* h, void* source, int32_t* out) {
    ChainBase* c = H(h);
    ChainBase* src = H(source);
    return Guard([&]() {
        gRandom = &c->rng;
        c->rng.Begin(0xffffffffu);
        c->RestoreRandom(&src->tree);
        c->step = src->step;
        if (out) out[0] = c->TotalSteps();
        return 0;
    });
}

int ref_chain_force_step(void* h, const double* x) {
    ChainBase* c = H(h);
    return Guard([&]() {
        Vector v(x, x + c->dim);
        c->Prop().ForceStep(v);
        return 0;
    });
}

int ref_chain_set_scan(void* h, int dim) {
    return Guard([&]() { H(h)->Prop().SetScanDimension(dim); return 0; });
}

int ref_chain_set_center(void* h, const double* v) {
    ChainBase* c = H(h);
    return Guard([&]() {
        Vector p(v, v + c->dim);
        return c->Prop().SetEstimatedCenter(p) ? 0 : -1;
    });
}

int ref_chain_update_proposal(void* h) {
    return Guard([&]() { H(h)->Prop().UpdateProposal(); return 0; });
}

int ref_chain_reset_proposal(void* h) {
    return Guard([&]() { H(h)->Prop().ResetProposal(); return 0; });
}

int ref_chain_get_state(void* h, double* s, double* accepted, double* center,
                        double* cov, double* decomp) {
    ChainBase* c = H(h);
    if (c->Vaat()) {
        // the sampler-level scalars; the proposal's own state comes from ref_chain_get_vaat
        if (s) {
            for (int k = 0; k < ORC_ST_COUNT; ++k) s[k] = 0.0;
            s[ORC_ST_SIGMA] = c->Vaat()->GetSigma();
            s[ORC_ST_ACCEPTANCE] = c->Vaat()->GetAcceptance();
            s[ORC_ST_ACCEPTANCE_WINDOW] = c->Vaat()->GetAcceptanceWindow();
            s[ORC_ST_ACCEPTANCE_RIGIDITY] = c->Vaat()->GetAcceptanceRigidity();
            s[ORC_ST_TRIALS] = c->Vaat()->GetTrials();
            s[ORC_ST_SUCCESSES] = c->Vaat()->GetSuccesses();
            s[ORC_ST_STEP_RMS] = c->StepRMS();
            s[ORC_ST_ACCEPTED_LLH] = c->AcceptedLlh();
            s[ORC_ST_PROPOSED_LLH] = c->ProposedLlh();
            s[ORC_ST_TOTAL_STEPS] = c->TotalSteps();
            s[ORC_ST_LLH_CALLS] = c->LlhCalls();
        }
        if (accepted) std::copy(c->Accepted().begin(), c->Accepted().end(), accepted);
        return 0;
    }
    TProposeAdaptiveStep& p = c->Prop();
    const int n = c->dim;
    if (s) {
        s[ORC_ST_SIGMA] = p.GetSigma();
        s[ORC_ST_ACCEPTANCE] = p.GetAcceptance();
        s[ORC_ST_ACCEPTANCE_TRIALS] = p.GetAcceptanceTrials();
        s[ORC_ST_ACCEPTANCE_WINDOW] = p.GetAcceptanceWindow();
        s[ORC_ST_ACCEPTANCE_RIGIDITY] = p.GetAcceptanceRigidity();
        s[ORC_ST_TARGET_ACCEPTANCE] = p.GetTargetAcceptance();
        s[ORC_ST_TRIALS] = p.GetTrials();
        s[ORC_ST_SUCCESSES] = p.GetSuccesses();
        s[ORC_ST_NEXT_UPDATE] = p.GetNextUpdate();
        s[ORC_ST_COVARIANCE_TRIALS] = p.GetCovarianceTrials();
        s[ORC_ST_COVARIANCE_WINDOW] = p.GetCovarianceWindow();
        s[ORC_ST_CENTER_TRIALS] = p.GetEstimatedCenterTrials();
        s[ORC_ST_COVARIANCE_TRACE] =
            p.fCurrentCov.GetNrows() == n ? p.GetCovarianceTrace() : 0.0;
        s[ORC_ST_SIGMA_TRACE] = p.fSigmaTrace;
        s[ORC_ST_STEP_RMS] = c->StepRMS();
        s[ORC_ST_ACCEPTED_LLH] = c->AcceptedLlh();
        s[ORC_ST_PROPOSED_LLH] = c->ProposedLlh();
        s[ORC_ST_TOTAL_STEPS] = c->TotalSteps();
        s[ORC_ST_LLH_CALLS] = c->LlhCalls();
    }
    if (accepted) std::copy(c->Accepted().begin(), c->Accepted().end(), accepted);
    if (center) std::copy(p.GetEstimatedCenter().begin(), p.GetEstimatedCenter().end(), center);
    if (cov && p.fCurrentCov.GetNrows() == n)
        std::copy(p.fCurrentCov.GetMatrixArray(), p.fCurrentCov.GetMatrixArray() + (size_t)n * n, cov);
    if (decomp && p.fDecomposition.GetNrows() == n)
        std::copy(p.fDecomposition.GetMatrixArray(), p.fDecomposition.GetMatrixArray() + (size_t)n * n, decomp);
    return 0;
}

double ref_chain_llh(void* h, const double* x) {
    ChainBase* c = H(h);
    Vector p(x, x + c->dim);
    return c->Llh(p);
}

int ref_chain_fake_hist(void* h, const double* x, double* out150) {
    if (H(h)->Fake2()) return ref_ex2_hist(H(h)->Fake2(), x, H(h)->dim, out150);
    FakeLikelihood* like = H(h)->Fake();
    if (!like) { gLastError = "not a FakeLikelihood chain"; return -1; }
    std::vector<double> p(x, x + H(h)->dim);
    like->FillHistograms(p);
    for (int b = 0; b < 50; ++b) {
        out150[b] = like->SimulatedClose->GetBinContent(b + 1);
        out150[50 + b] = like->SimulatedSeparated->GetBinContent(b + 1);
        out150[100 + b] = like->SimulatedDecayTag->GetBinContent(b + 1);
    }
    return 0;
}

// TDummyLogLikelihood::Covariance / Error as built by the reference's Init()
// (TDummyLogLikelihood.H:44-142); both are 100 x 100, row-major.
int ref_dummy_matrices(double* covariance, double* error) {
    if (TDummyLogLikelihood::Error.GetNrows() != 100) {
        TDummyLogLikelihood like;
        std::streambuf* old = std::cout.rdbuf(0);
        like.Init();
        std::cout.rdbuf(old);
    }
    if (covariance) std::copy(TDummyLogLikelihood::Covariance.GetMatrixArray(),
                              TDummyLogLikelihood::Covariance.GetMatrixArray() + 10000, covariance);
    if (error) std::copy(TDummyLogLikelihood::Error.GetMatrixArray(),
                         TDummyLogLikelihood::Error.GetMatrixArray() + 10000, error);
    return 0;
}

// The reference's own toy-input generators (example/Simulated.H:17-53 and
// example/FakeData.H:32-117) run under a seeded shim generator; used to check
// that the product's synthetic-input builder follows the same distributions.
long ref_fake_generate(unsigned long seed, int dataSignal, int dataBackground,
                       double oversample, orc_event* outEvents, long capacity,
                       double* outData150, double* outExposure) {
    TRandom* saved = gRandom;
    TRandom3 local(seed);
    gRandom = &local;
    FakeLikelihood like;
    std::streambuf* old = std::cout.rdbuf(0);
    like.Init(dataSignal, dataBackground, oversample);
    std::cout.rdbuf(old);
    gRandom = saved;
    long n = (long)like.SimulatedSample.size();
    if (n > capacity) n = capacity;
    if (outEvents) std::memcpy((void*)outEvents, like.SimulatedSample.data(), sizeof(orc_event) * n);
    if (outData150) {
        for (int b = 0; b < 50; ++b) {
            outData150[b] = like.DataClose->GetBinContent(b + 1);
            outData150[50 + b] = like.DataSeparated->GetBinContent(b + 1);
            outData150[100 + b] = like.DataDecayTag->GetBinContent(b + 1);
        }
    }
    if (outExposure) *outExposure = like.Corrections.ExposureRatio;
    return (long)like.SimulatedSample.size();
}

}  // extern "C"

// ---------------------------------------------------------------------------
// TSimpleHMC
// ---------------------------------------------------------------------------
namespace {
struct HmcBase {
    InjectedRandom rng;
    uint32_t step;
    int dim;
    HmcBase(uint64_t seed, uint32_t chain, int d) : rng(seed, chain), step(0), dim(d) {}
    virtual ~HmcBase() {}
    virtual void Set(int field, double v) = 0;
    virtual void Start(const Vector& x) = 0;
    virtual void Step(int type) = 0;
    virtual void State(double* s, double* acc, double* mom, double* cen, double* avg, double* cov, double* err) = 0;
    virtual double AcceptedPotential() = 0;
    virtual const Vector& Accepted() = 0;
    virtual double MeanEpsilon() = 0;
    virtual int LeapFrog() = 0;
};
template <class L, class G>
struct Hmc : public HmcBase {
    sMCMC::TSimpleHMC<L, G> hmc;
    Hmc(uint64_t seed, uint32_t chain, int d) : HmcBase(seed, chain, d), hmc(NULL) {}
    void Set(int field, double v) {
        if (field == ORC_HMC_ALPHA) hmc.SetAlpha(v);
        else if (field == ORC_HMC_MEAN_EPSILON) hmc.SetMeanEpsilon(v);
        else if (field == ORC_HMC_LEAPFROG) hmc.SetLeapFrog((int)v);
    }
    void Start(const Vector& x) { hmc.Start(x, false); }
    void Step(int type) { hmc.Step(false, type); }
    double AcceptedPotential() { return hmc.fAcceptedPotential; }
    const Vector& Accepted() { return hmc.fAccepted; }
    double MeanEpsilon() { return hmc.fMeanEpsilon; }
    int LeapFrog() { return hmc.fLeapFrogSteps; }
    void State(double* s, double* acc, double* mom, double* cen, double* avg, double* cov, double* err) {
        const int n = dim;
        if (s) {
            s[ORC_HS_ACCEPTANCE] = hmc.fCurrentAcceptance;
            s[ORC_HS_MEAN_EPSILON] = hmc.fMeanEpsilon;
            s[ORC_HS_LEAPFROG] = hmc.fLeapFrogSteps;
            s[ORC_HS_REVERSAL_LEN] = hmc.fReversalLen;
            s[ORC_HS_ACCEPTED_POTENTIAL] = hmc.fAcceptedPotential;
            s[ORC_HS_PROPOSED_POTENTIAL] = hmc.fProposedPotential;
            s[ORC_HS_CENTRAL_POTENTIAL] = hmc.fCentralPotential;
            s[ORC_HS_POTENTIAL_COUNT] = hmc.fPotentialCount;
            s[ORC_HS_GRADIENT_COUNT] = hmc.fPotentialGradientCount;
            s[ORC_HS_STEP_COUNT] = hmc.fStepCount;
            s[ORC_HS_COV_TRIALS] = hmc.fCovarianceTrials;
            s[ORC_HS_AVERAGE_TRIALS] = hmc.fAveragePointTrials;
            s[ORC_HS_EST_COV_TRACE] = hmc.fEstimatedCovarianceTrace;
            s[ORC_HS_CUR_COV_TRACE] = hmc.fCurrentCovarianceTrace;
            s[ORC_HS_ORBIT_LENGTH] = hmc.fEstimatedOrbitLength;
            s[ORC_HS_STEPS_REMAINING] = hmc.fStepsRemaining;
            s[ORC_HS_STEPS_SINCE_UPDATE] = hmc.fStepsSinceUpdate;
        }
        if (acc) std::copy(hmc.fAccepted.begin(), hmc.fAccepted.end(), acc);
        if (mom) std::copy(hmc.fAcceptedMomentum.begin(), hmc.fAcceptedMomentum.end(), mom);
        if (cen) std::copy(hmc.fCentralPoint.begin(), hmc.fCentralPoint.end(), cen);
        if (avg) std::copy(hmc.fAveragePoint.begin(), hmc.fAveragePoint.end(), avg);
        if (cov) std::copy(hmc.fEstimatedCovariance.GetMatrixArray(), hmc.fEstimatedCovariance.GetMatrixArray() + (size_t)n * n, cov);
        if (err) std::copy(hmc.fEstimatedError.GetMatrixArray(), hmc.fEstimatedError.GetMatrixArray() + (size_t)n * n, err);
    }
};
HmcBase* HH(void* h) { return static_cast<HmcBase*>(h); }
}  // namespace

extern "C" {

void* ref_hmc_create(int kind, int dim, int withGradient, uint64_t seed, uint32_t chain) {
    if (kind == ORC_LLH_DUMMY) {
        if (dim != 100) { gLastError = "reference TDummyLogLikelihood is 100-dim"; return 0; }
        if (TDummyLogLikelihood::Error.GetNrows() != 100) ref_dummy_matrices(0, 0);
        if (withGradient) return new Hmc<TDummyLogLikelihood, TDummyLogLikelihood>(seed, chain, 100);
        return new Hmc<TDummyLogLikelihood, SimpleHMCInvalidGradient>(seed, chain, 100);
    }
    if (kind == ORC_LLH_UNIT_GAUSS) return new Hmc<UnitGaussLikelihood, SimpleHMCInvalidGradient>(seed, chain, dim);
    if (kind == ORC_LLH_HORRIFIC && dim == 75) return new Hmc<THorrificLogLikelihood, THorrificLogLikelihood>(seed, chain, 75);
    if (kind == ORC_LLH_HARD && dim == 6) {
        if (withGradient) return new Hmc<THardLogLikelihood, THardLogLikelihood>(seed, chain, 6);
        return new Hmc<THardLogLikelihood, SimpleHMCInvalidGradient>(seed, chain, 6);
    }
    gLastError = "unsupported HMC likelihood";
    return 0;
}
void ref_hmc_destroy(void* h) { delete HH(h); }
int ref_hmc_set_error_matrix(void*, const double*, int) { gLastError = "the reference builds its own error matrix"; return -1; }
int ref_hmc_set(void* h, int field, double v) { HH(h)->Set(field, v); return 0; }
int ref_hmc_start(void* h, const double* x0) {
    HmcBase* c = HH(h);
    return Guard([&]() {
        gRandom = &c->rng;
        Vector x(x0, x0 + c->dim);
        c->Start(x);
        return 1;
    });
}
int ref_hmc_step(void* h, int nsteps, int type, double* potential, double* x, double* epsilon, int32_t* leapfrog) {
    HmcBase* c = HH(h);
    return Guard([&]() {
        gRandom = &c->rng;
        for (int s = 0; s < nsteps; ++s) {
            c->rng.Begin(c->step++);
            c->Step(type);
            if (potential) potential[s] = c->AcceptedPotential();
            if (epsilon) epsilon[s] = c->MeanEpsilon();
            if (leapfrog) leapfrog[s] = c->LeapFrog();
            if (x) std::copy(c->Accepted().begin(), c->Accepted().end(), x + (size_t)s * c->dim);
        }
        return 0;
    });
}
int ref_hmc_get_state(void* h, double* s, double* acc, double* mom, double* cen, double* avg, double* cov, double* err) {
    HH(h)->State(s, acc, mom, cen, avg, cov, err);
    return 0;
}

}  // extern "C"
