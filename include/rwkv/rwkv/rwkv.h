// rwkv.h — host API of the B200 RWKV-v4 uint8 engine: `RWKV`, `RWKVState`, the tensor table.
//
// Source-compatible with the reference's host header (harrisonvanderbyl/rwkv-cpp-accelerated
// include/rwkv/rwkv/rwkv.h): same class names, public members, method signatures, error
// messages and stdout prints, so examples/storygen/storygen.cpp, examples/terminalchat/chat.cpp
// and examples/vectordb/vectordb.cpp compile unchanged against `-I<repo>/include` and link
// against librwkv_b200.so (or the static librwkv_cuda.a alias).
//
// What is different underneath (see DESIGN.md):
//   * all compute goes through the C ABI in rwkv_b200.h (opaque handle) instead of the
//     reference's six C++-linkage backend hooks with 47 raw pointers (R.h:63-122);
//   * the recurrent state and the embedding table are resident in HBM. The host arrays of
//     `RWKVState` are mirrors: the live state is pulled from the device only when it is
//     read through this API (copy / getSubState / setSubState / syncToHost) and pushed only
//     after it was changed through this API. Set `RWKV::strictState = true` (or the
//     environment variable RWKV_B200_STRICT_STATE=1) to get the reference's exact behaviour
//     of copying the full state host->device before and device->host after every forward
//     (R.h:353,372) — needed only by code that pokes `state->statexx[i]` directly;
//   * everything is `inline`, so more than one translation unit may include this header
//     (the reference allows exactly one).
#if !defined(RWKV_H)
#define RWKV_H
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>

#include "rwkv/enums/enum.h"
#include "rwkv/rwkv/format.h"
#include "rwkv/sampler/typical.h"
#include "rwkv_b200.h"

// ---- tensor table (R.h:10-56, 84, 124-138), generated from format.h ----------------------------
namespace rwkv_detail {
struct NameTable {
    std::string v[rwkv_format::kNumTensors];
    NameTable() {
        for (int i = 0; i < rwkv_format::kNumTensors; ++i) v[i] = rwkv_format::name(i);
    }
};
struct TypeTable {
    unsigned long v[rwkv_format::kNumTensors];
    constexpr TypeTable() : v() {
        for (int i = 0; i < rwkv_format::kNumTensors; ++i) v[i] = (unsigned long)rwkv_format::kSpecs[i].dtype;
    }
};
inline NameTable g_names;
inline constexpr TypeTable g_types{};
} // namespace rwkv_detail

// names[i] / types[i]: printable name and element size in bytes of tensor-table slot i.
inline std::string (&names)[rwkv_format::kNumTensors] = rwkv_detail::g_names.v;
inline const unsigned long (&types)[rwkv_format::kNumTensors] = rwkv_detail::g_types.v;

// Element count of tensor i for a model with `a` layers and `b` embedding channels.
inline unsigned long long getSize(unsigned long long i, unsigned long long a, unsigned long long b) {
    return rwkv_format::elems((int)i, a, b);
}
inline unsigned long long Mtypes(unsigned long long i) { return types[i]; }
inline const char *getName(unsigned long long i) { return names[i].c_str(); }

// ---- RWKVState (R.h:140-242) ---------------------------------------------------------------------
// Five host arrays of num_layers*num_embed*stateSize doubles. Zero-initialised; deep copies.
class RWKVState {
  public:
    double *statexy;
    double *stateaa;
    double *statebb;
    double *statepp;
    double *statedd;
    unsigned long long num_layers;
    unsigned long long num_embed;
    unsigned long long stateSize;

    RWKVState(unsigned long long num_layers, unsigned long long num_embed, unsigned long long stateSize)
        : num_layers(num_layers), num_embed(num_embed), stateSize(stateSize) {
        allocate();
        for (double *a : {statexy, stateaa, statebb, statepp, statedd}) std::fill(a, a + count(), 0.0);
    }

    RWKVState(const RWKVState &other)
        : num_layers(other.num_layers), num_embed(other.num_embed), stateSize(other.stateSize) {
        other.syncToHost();
        allocate();
        copyFrom(other, 0, 0, count());
    }

    // One slot of `other` as a stateSize == 1 state. The reference indexes other[i + offset]
    // without the slot stride (R.h:205-209) while setSubState strides by num_layers*num_embed
    // (R.h:234-238); both agree for offset 0, the only value any caller uses. This
    // implementation uses the slot stride in both directions.
    RWKVState(const RWKVState &other, unsigned long long offset)
        : num_layers(other.num_layers), num_embed(other.num_embed), stateSize(1) {
        other.syncToHost();
        allocate();
        copyFrom(other, 0, offset * num_layers * num_embed, count());
    }

    RWKVState &operator=(const RWKVState &other) {
        if (this == &other) return *this;
        other.syncToHost();
        if (count() != other.count()) {
            release();
            num_layers = other.num_layers;
            num_embed = other.num_embed;
            stateSize = other.stateSize;
            allocate();
        }
        copyFrom(other, 0, 0, count());
        hostAhead = true;
        deviceAhead = false;
        return *this;
    }

    ~RWKVState() { release(); }

    // Get a substate
    RWKVState getSubState(unsigned long long offset = 0) {
        if (offset >= stateSize) {
            throw std::runtime_error("State get offset out of bounds, max offset is " + std::to_string(stateSize));
        }
        return RWKVState(*this, offset);
    }

    // Set a substate
    void setSubState(RWKVState &other, unsigned long long offset = 0) {
        if (offset >= stateSize) {
            throw std::runtime_error("State set offset out of bounds, max offset is " + std::to_string(stateSize));
        }
        other.syncToHost();
        if (stateSize > 1) syncToHost(); // the other slots must be current before a partial overwrite
        const unsigned long long n = num_layers * num_embed;
        copyFrom(other, offset * n, 0, n);
        deviceAhead = false;
        hostAhead = true;
    }

    // ---- device mirror protocol (not in the reference) ----------------------------------
    // Make the host arrays current (no-op unless this is the live state of a loaded RWKV
    // and a forward ran since the last pull).
    void syncToHost() const {
        if (engine && deviceAhead) {
            if (rwkv_b200_state_download(engine, statexy, stateaa, statebb, nullptr, statedd, stateSize) != 0)
                throw std::runtime_error(std::string("RWKV state download failed: ") + rwkv_b200_last_error());
            deviceAhead = false;
        }
    }
    // Tell the engine the host arrays were edited in place (e.g. state->stateaa[i] = ...).
    void markHostModified() { hostAhead = true; }

    rwkv_b200_model *engine = nullptr; // set only on the live state owned by an RWKV
    mutable bool deviceAhead = false;  // device holds a newer state than the host arrays
    bool hostAhead = false;            // host arrays must be uploaded before the next forward

  private:
    unsigned long long count() const { return num_layers * num_embed * stateSize; }
    void allocate() {
        const size_t bytes = (size_t)count() * sizeof(double);
        statexy = (double *)rwkv_b200_host_alloc(bytes);
        stateaa = (double *)rwkv_b200_host_alloc(bytes);
        statebb = (double *)rwkv_b200_host_alloc(bytes);
        statepp = (double *)rwkv_b200_host_alloc(bytes);
        statedd = (double *)rwkv_b200_host_alloc(bytes);
        if (!statexy || !stateaa || !statebb || !statepp || !statedd) throw std::bad_alloc();
    }
    void release() {
        for (double *a : {statexy, stateaa, statebb, statepp, statedd}) rwkv_b200_host_free(a);
        statexy = stateaa = statebb = statepp = statedd = nullptr;
    }
    void copyFrom(const RWKVState &o, unsigned long long dst_off, unsigned long long src_off, unsigned long long n) {
        std::copy(o.statexy + src_off, o.statexy + src_off + n, statexy + dst_off);
        std::copy(o.stateaa + src_off, o.stateaa + src_off + n, stateaa + dst_off);
        std::copy(o.statebb + src_off, o.statebb + src_off + n, statebb + dst_off);
        std::copy(o.statepp + src_off, o.statepp + src_off + n, statepp + dst_off);
        std::copy(o.statedd + src_off, o.statedd + src_off + n, statedd + dst_off);
    }
};

#include "rwkv/tokenizer/tokenizer.h"

// ---- RWKV (R.h:245-429) ---------------------------------------------------------------------------
class RWKV {
  public:
    // Tensor pointers (device pointers, see rwkv_b200_tensor). Valid after loadFile.
    int **tensors = new int *[rwkv_format::kNumTensors]();

    // Number of layers in model
    unsigned long long num_layers = 0;

    // Number of elements per embedding
    unsigned long long num_embed = 0;

    // Cpu tensor for reading logits (pinned; owned by the engine; writable, e.g. out[0] = -99)
    float *out = nullptr;

    unsigned long long maxContext = 1;

    // Cpu state tensors
    RWKVState *state = nullptr;

    GPT2Tokenizer *tokenizer = nullptr;

    bool ready = false;

    // Compatibility aliases of state->statexx
    double *statexy = nullptr;
    double *stateaa = nullptr;
    double *statebb = nullptr;
    double *statepp = nullptr;
    double *statedd = nullptr;

    // B200 engine handle and options (not in the reference)
    rwkv_b200_model *engine = nullptr;
    bool strictState = false; // true: full state H2D before / D2H after every forward (R.h:353,372)
    int device = 0;
    bool quietLoad = false;

    RWKV() {
        if (const char *e = std::getenv("RWKV_B200_STRICT_STATE")) strictState = std::atoi(e) != 0;
        if (const char *e = std::getenv("RWKV_B200_DEVICE")) device = std::atoi(e);
        if (const char *e = std::getenv("RWKV_B200_QUIET")) quietLoad = std::atoi(e) != 0;
    }
    RWKV(const RWKV &) = delete; // owns a device model; the examples' `RWKV Rwkv = RWKV();` is elided in C++17
    RWKV &operator=(const RWKV &) = delete;

    // Load from .bin file
    void loadFile(const std::string &filename, unsigned long long maxGPT = 1) {
        if (ready) {
            throw std::runtime_error("RWKV already loaded");
        }
        const int rc = rwkv_b200_load(filename.c_str(), maxGPT, device, quietLoad ? 1 : 0, &engine, &num_layers, &num_embed);
        if (rc == 2) { // the reference prints and exits when the file cannot be opened (R.cu:641-645)
            std::cout << "Error opening file " << filename << std::endl;
            std::exit(1);
        }
        if (rc != 0) {
            throw std::runtime_error(std::string("RWKV load failed: ") + rwkv_b200_last_error());
        }
        for (int i = 0; i < rwkv_format::kNumTensors; ++i) tensors[i] = (int *)rwkv_b200_tensor(engine, i);

        state = new RWKVState(num_layers, num_embed, maxGPT);
        state->engine = engine;

        // Deprecated, compatibility layer
        statexy = state->statexy;
        stateaa = state->stateaa;
        statebb = state->statebb;
        statepp = state->statepp;
        statedd = state->statedd;

        out = rwkv_b200_logits_host(engine);
        std::fill(out, out + RWKV_B200_VOCAB * maxGPT, 0.0f);

        maxContext = maxGPT;
        ready = true;
    }

    void loadTokenizer(std::string vocabPath) {
        auto _tokenizer = GPT2Tokenizer::load(vocabPath + "/vocab.json", vocabPath + "/merges.txt");
        if (!_tokenizer.has_value()) {
            std::cerr << "Failed to load tokenizer" << std::endl;
            return;
        }
        tokenizer = new GPT2Tokenizer(_tokenizer.value());
    }

    // Get number of elements in a tensor
    unsigned long long getTensorSize(unsigned long long i) { return getSize(i, num_layers, num_embed); }

    // Get the bytesize of a tensor
    unsigned long long getTensorTypes(unsigned long long i) { return types[i]; }

    float *forward(std::vector<unsigned long long> token, MODE mode) {
        if (!ready) {
            throw std::runtime_error("RWKV not loaded");
        }
        if (token.size() > maxContext) {
            throw std::runtime_error("Context too large, max context is " + std::to_string(maxContext));
        }
        if (token.empty()) return out;

        // host -> device only when the host copy is the newer one
        if (strictState || state->hostAhead) {
            const unsigned long long slots = strictState ? (unsigned long long)token.size() : state->stateSize;
            if (rwkv_b200_state_upload(engine, state->statexy, state->stateaa, state->statebb, nullptr, state->statedd,
                                       std::min(slots, state->stateSize)) != 0)
                throw std::runtime_error(std::string("RWKV state upload failed: ") + rwkv_b200_last_error());
            state->hostAhead = false;
        }
        if (rwkv_b200_forward(engine, token.data(), token.size(), mode == PARRALEL ? RWKV_B200_MODE_PARRALEL : RWKV_B200_MODE_GPT,
                              out) != 0)
            throw std::runtime_error(std::string("RWKV forward failed: ") + rwkv_b200_last_error());
        state->deviceAhead = true;
        if (strictState) state->syncToHost();
        return out;
    }

    float *forward(unsigned long long token) { return forward(std::vector<unsigned long long>{token}, GPT); }

    float *forward(std::vector<long long> token, MODE mode) {
        std::vector<unsigned long long> token2(token.begin(), token.end());
        return forward(token2, mode);
    }

    // Extension (the reference has no counterpart): draw the next token from the logits of the LAST
    // forward exactly as `typical(out, temp, tau)` would - same distribution, same process-wide
    // generator, hence the same token sequence - but on the GPU, where the logits already are: the
    // host sampler costs 0.4 ms per token (50277 double exps), a fifth of the whole forward. The device
    // kernel reports how close the uniform is to an interval boundary; in that (1e-9) case the host
    // path decides with the same uniform, so the result is the host's token in every case.
    // Edits made to `out[]` on the host after the forward are NOT seen; use typical(out, ...) for that.
    int sample(float temp = 0.9f, float tau = 0.8f) {
        (void)tau; // no effect in the reference either (see rwkv/sampler/typical.h)
        if (!ready) throw std::runtime_error("RWKV not loaded");
        const double u = std::generate_canonical<double, 53>(rwkv_sampler_generator());
        unsigned long long tok = 0;
        double margin = 0.0;
        if (rwkv_b200_sample_typical(engine, temp, u, &tok, &margin) == 0 && margin >= 1e-9) return (int)tok;
        return typical_with_u(out, temp, u);
    }

    // Extension: free-running generation on the device (rwkv_b200_generate). Same tokens, same state and same
    // position of the process-wide generator as the loop `forward(token); token = sample(temp);` run n times, or
    // until it produces one of the `stop` ids - without a host round trip per token. Returns t1..tk; the state has
    // consumed token, t1, ..., t(k-1) and `out` holds the logits of the last forward.
    std::vector<unsigned long long> generate(unsigned long long token, unsigned long long n, float temp = 0.9f,
                                             std::vector<unsigned long long> stop = {}) {
        // The loop's uniforms, drawn from a copy of the generator; the generator itself advances by the steps that
        // ran (generate_canonical<double, 53> on mt19937_64 takes exactly one draw).
        std::mt19937_64 gen = rwkv_sampler_generator();
        std::vector<double> u(n);
        for (double &x : u) x = std::generate_canonical<double, 53>(gen);
        std::vector<unsigned long long> toks = runGenerate(token, n, RWKV_B200_GEN_TYPICAL, temp, u.data(), stop);
        rwkv_sampler_generator().discard(toks.size());
        return toks;
    }

    // Extension: the same for the greedy loop `forward(token); token = argmax(out);`.
    std::vector<unsigned long long> generateGreedy(unsigned long long token, unsigned long long n,
                                                   std::vector<unsigned long long> stop = {}) {
        return runGenerate(token, n, RWKV_B200_GEN_GREEDY, 1.0f, nullptr, stop);
    }

    RWKVState emptyState() { return {num_layers, num_embed, 1}; }

    long long loadContext(std::string input, bool progress = false) {
        std::vector<long long> initial = tokenizer->encode(input);
        if (initial.empty()) return 0;
        std::cout << initial[0] << ":token";
        for (size_t i = 0; i < initial.size(); i += maxContext) {
            auto mvec = std::vector<unsigned long long>(initial.begin() + i,
                                                        initial.begin() + (std::min((size_t)(i + maxContext), initial.size())));
            forward(mvec, GPT);
            if (progress) {
                std::cout << "\r";
                std::cout << int(float(i) / initial.size() * 100) << "%";
                std::flush(std::cout);
            }
        }
        return initial[initial.size() - 1];
    }

    // destructor
    ~RWKV() {
        if (ready) {
            delete state;
            rwkv_b200_free(engine);
        }
        delete[] tensors;
        delete tokenizer;
    }

  private:
    std::vector<unsigned long long> runGenerate(unsigned long long token, unsigned long long n, int how, float temp,
                                                const double *uniforms, const std::vector<unsigned long long> &stop) {
        if (!ready) throw std::runtime_error("RWKV not loaded");
        if (n == 0) return {};
        if (strictState || state->hostAhead) { // as in forward: one token on slot 0
            const unsigned long long slots = strictState ? 1ull : state->stateSize;
            if (rwkv_b200_state_upload(engine, state->statexy, state->stateaa, state->statebb, nullptr, state->statedd,
                                       std::min(slots, state->stateSize)) != 0)
                throw std::runtime_error(std::string("RWKV state upload failed: ") + rwkv_b200_last_error());
            state->hostAhead = false;
        }
        std::vector<unsigned long long> toks(n);
        unsigned long long k = 0;
        if (rwkv_b200_generate(engine, token, n, how, temp, uniforms, stop.data(), (int)stop.size(), toks.data(), &k, out) != 0)
            throw std::runtime_error(std::string("RWKV generate failed: ") + rwkv_b200_last_error());
        state->deviceAhead = true;
        if (strictState) state->syncToHost();
        toks.resize(k);
        return toks;
    }
};

#endif
