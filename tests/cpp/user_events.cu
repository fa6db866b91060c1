// user_events.cu -- an analysis program written against the mirror headers with
// its likelihood as a user EVENT functor (GaussEvents of user_events.cuh): the
// mean and width of a sample read from a file of doubles.
//   user_events chain <events.bin> <seed> <chain> <steps>   one chain, recorded in a TTree
//   user_events hmc <events.bin> <chains> <steps>           TSimpleHMC<GaussEvents>, finite differences
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "user_events.cuh"
#include "TSimpleHMC.H"

static std::vector<GaussEvents::Event> ReadEvents(const char* path) {
    std::vector<GaussEvents::Event> events;
    FILE* f = std::fopen(path, "rb");
    if (!f) throw std::runtime_error(std::string("cannot open ") + path);
    GaussEvents::Event e;
    while (std::fread(&e.v, sizeof(double), 1, f) == 1) events.push_back(e);
    std::fclose(f);
    return events;
}

static int Chain(const char* path, unsigned long long seed, int chain, int steps) {
    const std::vector<GaussEvents::Event> events = ReadEvents(path);
    TTree tree("Gauss", "Tree of accepted points");
    sMCMC::TSimpleMCMC<GaussEvents> mcmc(&tree);
    mcmc.SetSeed(seed);
    mcmc.SetDevice(0, chain);
    mcmc.SetEvents(events);                          // kept until Start creates the engine
    mcmc.GetProposeStep().SetDim(2);
    sMCMC::Vector p(2);
    p[0] = 2.5;
    p[1] = 1.5;
    if (!mcmc.Start(p, true)) return 2;
    const double host = smcmc_user::EventLikelihoodHost(mcmc.GetLogLikelihood(), events.data(), (int64_t)events.size(),
                                                        p.data(), 2);
    std::printf("start llh %.17g host %.17g\n", mcmc.GetAcceptedLogLikelihood(), host);
    for (int i = 0; i < steps; ++i) {
        if (i == steps / 2) mcmc.SetEvents(events);  // uploaded at once: the same sample again
        const bool ok = mcmc.Step();
        std::printf("step %d acc %d llh %.17g x %.17g %.17g\n", i, (int)ok, mcmc.GetAcceptedLogLikelihood(),
                    mcmc.GetAccepted()[0], mcmc.GetAccepted()[1]);
    }
    std::printf("entries %ld calls %d\n", tree.GetEntries(), mcmc.GetLogLikelihoodCount());
    return 0;
}

static int Hmc(const char* path, int chains, int steps) {
    const std::vector<GaussEvents::Event> events = ReadEvents(path);
    sMCMC::TSimpleHMC<GaussEvents> hmc;
    hmc.SetChains(chains);
    hmc.SetSeed(61);
    hmc.SetEvents(events);
    sMCMC::Vector p(2);
    p[0] = 2.8;
    p[1] = 2.1;
    hmc.Start(p, false);
    for (int i = 0; i < steps; ++i) hmc.Step(false, 1);
    int finite = 0;
    for (int c = 0; c < chains; ++c) finite += std::isfinite(hmc.GetAcceptedPotential(c)) ? 1 : 0;
    std::printf("hmc finite %d of %d potentials %d gradients %d\n", finite, chains, hmc.GetPotentialCount(),
                hmc.GetGradientCount());
    const sMCMC::Vector x = hmc.GetAccepted();
    std::printf("hmc x %.10g %.10g\n", x[0], x[1]);
    return 0;
}

int main(int argc, char** argv) {
    if (argc < 3) {
        std::fprintf(stderr, "usage: user_events chain <events.bin> <seed> <chain> <steps> | hmc <events.bin> <chains> <steps>\n");
        return 1;
    }
    try {
        if (!std::strcmp(argv[1], "hmc")) return Hmc(argv[2], argc > 3 ? std::atoi(argv[3]) : 64, argc > 4 ? std::atoi(argv[4]) : 50);
        return Chain(argv[2], argc > 3 ? std::strtoull(argv[3], nullptr, 10) : 1, argc > 4 ? std::atoi(argv[4]) : 0,
                     argc > 5 ? std::atoi(argv[5]) : 100);
    } catch (std::exception& e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
}
