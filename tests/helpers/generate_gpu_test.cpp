// generate_gpu_test.cpp — RWKV::generate(tok, n, temp) must give the tokens of the loop
//   forward(tok); tok = sample(temp);
// from the same generator state, and leave the process-wide generator where the loop leaves it (the next
// generate_canonical draw is equal): once for a full run, once with a stop id that ends the run early.
// usage: generate_gpu_test model.bin
#include <cstdio>
#include <string>
#include <vector>
#include "rwkv.h"

static void reset(RWKV &net) {
    RWKVState zero = net.emptyState();
    net.state->setSubState(zero, 0);
}

static int check(RWKV &net, float temp, unsigned long long n, std::vector<unsigned long long> stop, unsigned seed) {
    auto &gen = rwkv_sampler_generator();
    reset(net);
    gen.seed(seed);
    std::vector<unsigned long long> want;
    unsigned long long tok = 4118;
    for (unsigned long long i = 0; i < n; ++i) {
        net.forward(tok);
        tok = (unsigned long long)net.sample(temp);
        want.push_back(tok);
        if (std::find(stop.begin(), stop.end(), tok) != stop.end()) break;
    }
    const double next_want = std::generate_canonical<double, 53>(gen);
    std::vector<float> out_want(net.out, net.out + 50277);
    reset(net);
    gen.seed(seed);
    const std::vector<unsigned long long> got = net.generate(4118, n, temp, stop);
    const double next_got = std::generate_canonical<double, 53>(gen);
    if (got != want) {
        printf("FAIL temp %.1f: %zu tokens generated, %zu by the loop\n", temp, got.size(), want.size());
        for (size_t i = 0; i < std::min(got.size(), want.size()); ++i)
            if (got[i] != want[i]) {
                printf("  first difference at step %zu: %llu vs %llu\n", i, got[i], want[i]);
                break;
            }
        return 1;
    }
    if (next_got != next_want) {
        printf("FAIL temp %.1f: generator position differs after %zu steps\n", temp, got.size());
        return 1;
    }
    if (!std::equal(out_want.begin(), out_want.end(), net.out)) {
        printf("FAIL temp %.1f: RWKV::out is not the last forward's logits\n", temp);
        return 1;
    }
    printf("ok temp %.1f: %zu tokens\n", temp, got.size());
    return 0;
}

int main(int argc, char **argv) {
    if (argc < 2) return 2;
    setenv("RWKV_B200_QUIET", "1", 1);
    RWKV net;
    net.loadFile(argv[1]);
    for (float temp : {0.9f, 0.3f})
        if (check(net, temp, 40, {}, 77)) return 1;
    // a stop id taken from a full run: its first occurrence ends the run there
    auto &gen = rwkv_sampler_generator();
    reset(net);
    gen.seed(91);
    std::vector<unsigned long long> full = net.generate(4118, 40, 2.0f);
    size_t k = 8;
    while (k < full.size() && std::find(full.begin(), full.begin() + k, full[k]) != full.begin() + k) ++k;
    if (k >= full.size()) {
        printf("FAIL: no fresh token after step 8 to stop at\n");
        return 1;
    }
    if (check(net, 2.0f, 40, {full[k]}, 91)) return 1;
    reset(net);
    gen.seed(91);
    if (net.generate(4118, 40, 2.0f, {full[k]}).size() != k + 1) {
        printf("FAIL: the stop id did not end the run after %zu tokens\n", k + 1);
        return 1;
    }
    printf("ALL OK\n");
    return 0;
}
