// user_weighted.cu -- an analysis program written against the mirror headers with
// its likelihood as a user WEIGHTED binned event functor (GaussWeighted of
// user_weighted.cuh): the mean and width of a data histogram, fitted with a flat
// template reweighted event by event.
//   user_weighted <template.bin> <data40.bin> <seed> <chain> <steps>
// One chain recorded in a TTree; then the data histogram is doubled through
// GetLogLikelihood() and SyncLikelihood(), and the value at the start point is
// printed before and after.
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "user_weighted.cuh"
#include "TSimpleMCMC.H"

static std::vector<double> ReadDoubles(const char* path) {
    std::vector<double> v;
    FILE* f = std::fopen(path, "rb");
    if (!f) throw std::runtime_error(std::string("cannot open ") + path);
    double d;
    while (std::fread(&d, sizeof(double), 1, f) == 1) v.push_back(d);
    std::fclose(f);
    return v;
}

static double Value(sMCMC::TSimpleMCMC<GaussWeighted>& mcmc, const sMCMC::Vector& p) {
    double v = 0.0;
    if (smcmc_eval(mcmc.GetEngine(), p.data(), 1, &v) != SMCMC_OK) throw std::runtime_error("smcmc_eval");
    return v;
}

int main(int argc, char** argv) {
    if (argc < 3) {
        std::fprintf(stderr, "usage: user_weighted <template.bin> <data40.bin> [seed] [chain] [steps]\n");
        return 1;
    }
    try {
        std::vector<GaussWeighted::Event> events;
        for (double u : ReadDoubles(argv[1])) events.push_back(GaussWeighted::Event{u});
        const std::vector<double> data = ReadDoubles(argv[2]);
        if (data.size() != GaussWeighted::kBins) throw std::runtime_error("data histogram must have 40 bins");
        const unsigned long long seed = argc > 3 ? std::strtoull(argv[3], nullptr, 10) : 1;
        const int chain = argc > 4 ? std::atoi(argv[4]) : 0, steps = argc > 5 ? std::atoi(argv[5]) : 100;

        TTree tree("Gauss", "Tree of accepted points");
        sMCMC::TSimpleMCMC<GaussWeighted> mcmc(&tree);
        GaussWeighted& like = mcmc.GetLogLikelihood();
        like.dataTotal = 0.0;
        for (int b = 0; b < GaussWeighted::kBins; ++b) {
            like.data[b] = data[b];
            like.dataTotal += data[b];
        }
        mcmc.SetSeed(seed);
        mcmc.SetDevice(0, chain);
        mcmc.SetEvents(events);                      // kept until Start creates the engine
        mcmc.GetProposeStep().SetDim(2);
        sMCMC::Vector p(2);
        p[0] = 2.5;
        p[1] = 1.5;
        if (!mcmc.Start(p, true)) return 2;
        const double host =
            smcmc_user::WeightedBinnedLikelihoodHost(like, events.data(), (int64_t)events.size(), p.data(), 2);
        std::printf("start llh %.17g host %.17g\n", mcmc.GetAcceptedLogLikelihood(), host);
        for (int i = 0; i < steps; ++i) {
            const bool ok = mcmc.Step();
            std::printf("step %d acc %d llh %.17g x %.17g %.17g\n", i, (int)ok, mcmc.GetAcceptedLogLikelihood(),
                        mcmc.GetAccepted()[0], mcmc.GetAccepted()[1]);
        }
        std::printf("entries %ld calls %d\n", tree.GetEntries(), mcmc.GetLogLikelihoodCount());

        const double before = Value(mcmc, p);
        for (int b = 0; b < GaussWeighted::kBins; ++b) like.data[b] *= 2.0;
        like.dataTotal *= 2.0;
        const double stale = Value(mcmc, p);
        mcmc.SyncLikelihood();
        const double after = Value(mcmc, p);
        const double hostAfter =
            smcmc_user::WeightedBinnedLikelihoodHost(like, events.data(), (int64_t)events.size(), p.data(), 2);
        std::printf("sync before %.17g stale %.17g after %.17g host %.17g\n", before, stale, after, hostAfter);
        return 0;
    } catch (std::exception& e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
}
