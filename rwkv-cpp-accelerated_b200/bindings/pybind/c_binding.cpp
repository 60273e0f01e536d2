// c_binding.cpp — Python module `rwkv` with the reference's pybind surface
// (bindings/pybind/c_binding.cpp:158-175 there): the same eleven function names, argument
// order and return types, so bindings/pybind/binding.py, tests/test_pybind.py,
// examples/pybind-flask and examples/pybind-interactive-chat run unchanged.
//
// Differences from the reference binding, all of them fixes of defects SURVEY.md 8(b) lists:
//   * tokenizerEncode returns the tokenizer's std::vector<long long> as a Python list (the
//     reference declares std::vector<int64_t>, which does not compile on LP64 Linux);
//   * initState() zeroes the LIVE state (device + host mirror); the reference re-allocates
//     the compatibility aliases, which resets nothing (c_binding.cpp:41-60);
//   * getState() returns five float64 arrays of n_layers*n_embed elements copied from the
//     live state; the reference copies 50277 elements regardless of the model size
//     (c_binding.cpp:81-110, out of bounds for small models).
// Handles are the same opaque capsules (void*).
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include "rwkv.h"

namespace py = pybind11;

static void *initRwkv() { return new RWKV(); }

static void *initTokenizer(const std::string &vocab_filename, const std::string &merges_filename) {
    std::optional<GPT2Tokenizer> loaded = GPT2Tokenizer::load(vocab_filename, merges_filename);
    if (!loaded.has_value()) {
        std::cerr << "Failed to load tokenizer" << std::endl;
        throw py::value_error("Failed to load tokenizer");
    }
    return new GPT2Tokenizer(loaded.value());
}

static void initRwkvOutput(void *h) {
    RWKV *net = static_cast<RWKV *>(h);
    std::fill(net->out, net->out + 50277, 0.0f);
}

static void initRwkvState(void *h) {
    RWKV *net = static_cast<RWKV *>(h);
    RWKVState zero = net->emptyState();
    for (unsigned long long slot = 0; slot < net->state->stateSize; ++slot) net->state->setSubState(zero, slot);
}

static py::array_t<float> getRwkvOutput(void *h) {
    RWKV *net = static_cast<RWKV *>(h);
    py::array_t<float> out(50277);
    std::copy(net->out, net->out + 50277, out.mutable_data());
    return out;
}

static py::list getRwkvState(void *h) {
    RWKV *net = static_cast<RWKV *>(h);
    net->state->syncToHost();
    const size_t n = (size_t)(net->num_layers * net->num_embed);
    py::list result;
    for (const double *src : {net->state->statexy, net->state->stateaa, net->state->statebb, net->state->statepp,
                              net->state->statedd}) {
        py::array_t<double> a(n);
        std::copy(src, src + n, a.mutable_data());
        result.append(a);
    }
    return result;
}

static std::vector<long long> tokenizerEncode(void *h, std::string text) {
    return static_cast<GPT2Tokenizer *>(h)->encode(text);
}

static py::object tokenizerDecode(void *h, int token) {
    const std::string s = static_cast<GPT2Tokenizer *>(h)->decode({(long long)token});
    // byte-level tokens need not be valid UTF-8 on their own; pybind's std::string caster would throw
    PyObject *u = PyUnicode_DecodeUTF8(s.data(), (Py_ssize_t)s.size(), "replace");
    return py::reinterpret_steal<py::object>(u);
}

// Samples from the logits of the last modelForward. The Python side never gets a writable view of the
// internal logits (getOutput copies), so the device sampler gives exactly the host sampler's tokens here.
static int typicalSample(void *h, float temp = 0.9, float tau = 0.8) {
    return static_cast<RWKV *>(h)->sample(temp, tau);
}

// Not in the reference binding: RWKV::generate / generateGreedy (free-running generation on the device), the same
// tokens as modelForward + typicalSample (or + arg-max) in a loop.
static std::vector<unsigned long long> generate(void *h, int64_t token, int64_t n, float temp, std::vector<unsigned long long> stop,
                                                bool greedy) {
    if (token < 0 || n < 0) throw py::value_error("generate: token and n must be non-negative");
    RWKV *net = static_cast<RWKV *>(h);
    py::gil_scoped_release release;
    return greedy ? net->generateGreedy((unsigned long long)token, (unsigned long long)n, stop)
                  : net->generate((unsigned long long)token, (unsigned long long)n, temp, stop);
}

static std::tuple<int64_t, int64_t> loadWrapper(void *h, const std::string &filename) {
    RWKV *net = static_cast<RWKV *>(h);
    net->loadFile(filename);
    return std::make_tuple((int64_t)net->num_layers, (int64_t)net->num_embed);
}

static void modelForward(void *h, int64_t token) {
    RWKV *net = static_cast<RWKV *>(h);
    py::gil_scoped_release release; // the reference holds the GIL for the whole forward
    net->forward((unsigned long long)token);
}

PYBIND11_MODULE(rwkv, m) {
    m.def("initRwkv", &initRwkv, "initRwkv");
    m.def("modelForward", &modelForward, "rwkvc");
    m.def("loadModel", &loadWrapper, "load");

    m.def("initState", &initRwkvState, "initState");
    m.def("getState", &getRwkvState, "getRwkvState");

    m.def("initOutput", &initRwkvOutput, "initOutput");
    m.def("getOutput", &getRwkvOutput, "getRwkvOutput");

    m.def("initTokenizer", &initTokenizer, "initTokenizer");
    m.def("tokenizerEncode", &tokenizerEncode, "tokenizerEncode");
    m.def("tokenizerDecode", &tokenizerDecode, "tokenizerDecode");

    m.def("typicalSample", &typicalSample, "typicalSample", py::arg("handle"), py::arg("temp") = 0.9f, py::arg("tau") = 0.8f);
    m.def("generate", &generate, "generate", py::arg("handle"), py::arg("token"), py::arg("n"), py::arg("temp") = 0.9f,
          py::arg("stop") = std::vector<unsigned long long>{}, py::arg("greedy") = false);
}
