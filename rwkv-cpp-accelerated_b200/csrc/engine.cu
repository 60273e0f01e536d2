// engine.cu — host side of the B200 RWKV-v4 uint8 decode engine + the C ABI (include/rwkv_b200.h).
//
// Responsibilities:
//   * load a reference-format .bin (include/rwkv/cuda/rwkv.cu:638-717 semantics): each rank reads only
//     the slices of the matrices it streams, stages them through pinned memory, and repacks on the device
//     (transpose to [out][in], centre to s8, fold 128*r + o into one offset vector);
//   * keep state, embedding table, weights and logits resident in HBM;
//   * issue one token as ONE cooperative launch of the persistent token kernel (token_kernel.cuh);
//   * wire the exchange blocks of the ranks of a tensor-parallel group (CUDA IPC);
//   * measurement hooks used by bench.py.
//
// There is deliberately no CPU code path: every entry point that computes fails with an error when
// no sm_100 device is present.
#include <algorithm>
#include <cerrno>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cuda_runtime.h>

#include "../../include/rwkv/enums/enum.h"
#include "../../include/rwkv/sampler/typical.h"
#include "../../include/rwkv_b200.h"
#include "aux_kernels.cuh"
#include "binfmt.h"
#include "prefill.cuh"
#include "token_kernel.cuh"

namespace rk {
const void *token_entry_gen(int cpl, bool full); // generate_kernels.cu
}

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return fail(100 + (int)e__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__),  \
                        __FILE__, __LINE__);                                                       \
    } while (0)

const char *kKernelNames[1] = {"token"};

} // namespace

struct rwkv_b200_model {
    int device = 0;
    int sms = 0;
    int grid = 0;
    int cpl = 0;
    double *d_sample = nullptr, *h_sample = nullptr; // device sampler result {token, margin}
    // generate: device [cap] uniforms + [cap] tokens + [cap] margins, and a pinned host mirror of the same layout
    unsigned char *d_gen = nullptr, *h_gen = nullptr;
    unsigned long long gen_cap = 0;
    double sample_margin = 1e-9; // set_option "sample_margin": the device's sampled token is kept at or above it
    size_t xch_bytes = 0;   // exchange block (peer-visible with tensor parallelism)
    bool tp_wired = false;  // peers' exchange blocks imported
    std::vector<void *> ipc_opened;
    unsigned long long L = 0, E = 0, max_gpt = 1;
    cudaStream_t stream = nullptr;
    rk::Params p{};
    size_t smem = 0;
    std::vector<void *> allocs;
    void *tensors[RWKV_B200_NUM_TENSORS] = {};
    double *spp = nullptr; // state_pp lives on the device only to honour the tensor table
    rk::Ctrl *h_ctrl = nullptr; // pinned [max_gpt]
    float *h_logits = nullptr;  // pinned [max_gpt][V]
    unsigned long long *h_next = nullptr;
    rk::Diag *h_diag = nullptr; // mapped pinned: the kernel's last words before a timeout trap
    int max_layers = -1;        // debug: run only the first n layers
    unsigned long long launches = 0;
    unsigned int epoch = 0, tk = 0; // exchange epochs (token_kernel.cuh); identical on every rank
    int tp_rank = 0, tp_size = 1;
    rk::PrefillState pf{};
};

namespace {

using M = rwkv_b200_model;

template <class T> int dmalloc(M *m, T **out, size_t count) {
    void *p = nullptr;
    CK(cudaMalloc(&p, count * sizeof(T) + 256));
    m->allocs.push_back(p);
    *out = reinterpret_cast<T *>(p);
    return 0;
}

int layers_to_run(const M *m) { return m->max_layers >= 0 && m->max_layers < (int)m->L ? m->max_layers : (int)m->L; }

// A failed synchronisation: if the kernel left a diagnostic record, say what it was waiting for.
int sync_failed(M *m, cudaError_t e, const char *what) {
    const rk::Diag *d = m->h_diag;
    if (d && d->code) {
        static const char *names[] = {"", "slice statistics", "activation vector", "offset sums", "peer partial sums",
                                      "sigmoid exchange", "completion flags", "arg-max candidates", "ring (full)", "ring (empty)",
                                      "cluster: limb planes free", "cluster: limb planes written", "sampler partials"};
        return fail(100 + (int)e,
                    "%s failed: %s; token kernel timed out waiting for %s: rank %u cta %u thread %u layer %u kind %u "
                    "expected tag %u saw %u aux %llu (a peer rank that never launched, or a protocol bug)",
                    what, cudaGetErrorString(e), d->code < 13 ? names[d->code] : "?", d->rank, d->cta, d->thread, d->layer,
                    d->kind, d->expect, d->seen, d->aux);
    }
    return fail(100 + (int)e, "%s failed: %s", what, cudaGetErrorString(e));
}
#define SYNC(m)                                                          \
    do {                                                                 \
        cudaError_t e__ = cudaStreamSynchronize((m)->stream);            \
        if (e__ != cudaSuccess) return sync_failed((m), e__, "forward"); \
    } while (0)

// ---- kernel dispatch on the model width -------------------------------------------------
// CPL = 16-byte chunks per lane of an n_embed-byte row; FULL = n_embed == CPL * 512 (no tail predicates).
// gen: the instantiation of rwkv_b200_generate (no trace stamps; generate_kernels.cu)
const void *token_entry(int cpl, bool full, bool trace, bool gen = false) {
    if (gen) return rk::token_entry_gen(cpl, full);
#define X(A)                                                                                                          \
    if (cpl == A) {                                                                                                   \
        if (trace) return full ? (const void *)rk::k_token<A, true, true> : (const void *)rk::k_token<A, false, true>; \
        return full ? (const void *)rk::k_token<A, true, false> : (const void *)rk::k_token<A, false, false>;          \
    }
    RK_CPLS(X)
#undef X
    return nullptr;
}

int chunks_per_lane(unsigned long long seg_bytes) {
    int c = (int)((seg_bytes + 511) / 512);
    if (c < 2) c = 2;
    return (c + 1) & ~1;
}

// Ring geometry: a tile is eight row segments of n_embed bytes (one per consumer warp); as many stages
// as fit beside the limb planes.
void configure_ring(M *m) {
    rk::Params &p = m->p;
    p.tile_bytes = (int)(8 * m->E);
    p.stages = (int)std::min<size_t>(rk::kMaxStages, (rk::kSmemLimit - rk::smem_bytes(0, 0, p.plane_cap)) / p.tile_bytes);
    m->smem = rk::smem_bytes(p.stages, p.tile_bytes, p.plane_cap);
}

void fill_launch(int grid, int cluster, size_t smem, cudaLaunchConfig_t &cfg, cudaLaunchAttribute (&attrs)[2], cudaStream_t s) {
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(rk::kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    attrs[0].id = cudaLaunchAttributeCooperative;
    attrs[0].val.cooperative = 1;
    attrs[1].id = cudaLaunchAttributeClusterDimension;
    attrs[1].val.clusterDim.x = (unsigned int)cluster;
    attrs[1].val.clusterDim.y = 1;
    attrs[1].val.clusterDim.z = 1;
    cfg.attrs = attrs;
    cfg.numAttrs = cluster > 1 ? 2 : 1;
}

int launch_token(M *m, int feed, bool greedy, const unsigned long long *stream, cudaStream_t s, bool gen = false) {
    if (m->tp_size > 1 && !m->tp_wired)
        return fail(7, "tensor parallelism: call rwkv_b200_tp_import with every rank's handle before the first forward");
    rk::Params prm = m->p;
    prm.L_run = layers_to_run(m);
    prm.feed_mode = feed;
    prm.greedy = greedy ? 1 : 0;
    prm.stream = stream;
    prm.ep0 = m->epoch;
    prm.tk = ++m->tk;
    if (prm.tk == 0) prm.tk = ++m->tk; // tag 0 means "never written"
    m->epoch += (unsigned int)prm.L_run + 1u;
    void *args[] = {&prm};
    const bool full = m->E == (unsigned long long)m->cpl * 512ull;
    const void *fn = token_entry(m->cpl, full, m->p.trace != nullptr, gen);
    if (!fn) return fail(3, "no kernel for %d chunks per lane", m->cpl);
    // cooperative: all CTAs resident together (they wait for each other's words); clusters of p.cluster CTAs share
    // the gather through distributed shared memory
    cudaLaunchConfig_t cfg{};
    cudaLaunchAttribute attrs[2];
    fill_launch(m->grid, m->p.cluster, m->smem, cfg, attrs, s);
    CK(cudaLaunchKernelExC(&cfg, fn, args));
    m->launches += 1;
    return 0;
}

// ---- loader --------------------------------------------------------------------------------
struct FileReader {
    int fd = -1;
    uint8_t *pin = nullptr;
    size_t pin_bytes = 0;
    ~FileReader() {
        if (fd >= 0) close(fd);
        if (pin) cudaFreeHost(pin);
    }
};

int read_exact(int fd, void *dst, size_t n, uint64_t off) {
    uint8_t *d = (uint8_t *)dst;
    while (n) {
        ssize_t got = pread(fd, d, n, (off_t)off);
        if (got < 0) {
            if (errno == EINTR) continue;
            return fail(4, "read error: %s", strerror(errno));
        }
        if (got == 0) return fail(4, "model file truncated");
        d += got;
        off += (uint64_t)got;
        n -= (size_t)got;
    }
    return 0;
}

// `rows` file rows of `row_stride` bytes starting at `off`; of each row the bytes [col0, col0 + cols)
// -> device dst, packed [rows][cols], through the pinned staging buffer. A rank of a tensor-parallel
// group reads only the columns / rows it streams.
int upload_rows(M *m, FileReader &fr, uint64_t off, size_t rows, size_t row_stride, size_t col0, size_t cols, void *dst) {
    uint8_t *d = (uint8_t *)dst;
    if (cols == row_stride) { // whole rows: one contiguous byte range
        size_t n = rows * cols;
        while (n) {
            const size_t c = std::min(n, fr.pin_bytes);
            int rc = read_exact(fr.fd, fr.pin, c, off);
            if (rc) return rc;
            CK(cudaMemcpyAsync(d, fr.pin, c, cudaMemcpyHostToDevice, m->stream));
            CK(cudaStreamSynchronize(m->stream));
            d += c;
            off += c;
            n -= c;
        }
        return 0;
    }
    if (cols > fr.pin_bytes) return fail(4, "row slice of %zu bytes exceeds the staging buffer", cols);
    const size_t per = fr.pin_bytes / cols;
    for (size_t r = 0; r < rows; r += per) {
        const size_t n = std::min(per, rows - r);
        for (size_t i = 0; i < n; ++i) {
            int rc = read_exact(fr.fd, fr.pin + i * cols, cols, off + (r + i) * row_stride + col0);
            if (rc) return rc;
        }
        CK(cudaMemcpyAsync(d + r * cols, fr.pin, n * cols, cudaMemcpyHostToDevice, m->stream));
        CK(cudaStreamSynchronize(m->stream));
    }
    return 0;
}

template <class T> int upload_tensor(M *m, FileReader &fr, int tid, T **out) {
    const size_t n = binfmt::elems(tid, m->L, m->E);
    int rc = dmalloc(m, out, n);
    if (rc) return rc;
    return upload_rows(m, fr, binfmt::offset(tid, m->L, m->E), 1, n * sizeof(T), 0, n * sizeof(T), *out);
}

// uint8 matrix family `tid`: `mats` matrices stored [rows_in][cols_out]; this rank keeps input rows
// [in0, in0 + nin) and output columns [out0, out0 + nout) -> int8 [nout][nin] per matrix.
int upload_matrix(M *m, FileReader &fr, int tid, size_t mats, size_t rows_in, size_t cols_out, size_t in0, size_t nin,
                  size_t out0, size_t nout, uint8_t *d_raw, int8_t **out) {
    int rc = dmalloc(m, out, mats * nin * nout);
    if (rc) return rc;
    const uint64_t base = binfmt::offset(tid, m->L, m->E);
    for (size_t i = 0; i < mats; ++i) {
        rc = upload_rows(m, fr, base + i * rows_in * cols_out + in0 * cols_out, nin, cols_out, out0, nout, d_raw);
        if (rc) return rc;
        dim3 g((unsigned)((nout + 63) / 64), (unsigned)((nin + 63) / 64));
        rk::k_transpose_xor<<<g, 256, 0, m->stream>>>(d_raw, nout, (int)nin, (int)nout, *out + i * nin * nout, nin, 0);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(m->stream));
    }
    return 0;
}

int centre(M *m, const float *r, const float *o, size_t n, const float **out) {
    float *oc = nullptr;
    int rc = dmalloc(m, &oc, n);
    if (rc) return rc;
    rk::k_centre_offsets<<<(unsigned)((n + 255) / 256), 256, 0, m->stream>>>(r, o, oc, n);
    CK(cudaGetLastError());
    *out = oc;
    return 0;
}

// Capacity checks of the per-CTA shared arrays for a grid of `grid` CTAs.
bool grid_fits(unsigned long long E, unsigned long long Er, unsigned long long Vr, int grid) {
    const unsigned long long g = (unsigned long long)grid;
    const unsigned long long ne = (E + g - 1) / g + 1, nc = (Er + g - 1) / g + 1, nk = (4 * Er + g - 1) / g + 1, nv = (Vr + g - 1) / g + 1;
    return grid >= 1 && grid <= rk::kMaxGrid && E >= g && ne <= (unsigned long long)rk::kMaxSlice &&
           nk <= 160 && nk + nc <= (unsigned long long)rk::kMaxRowsPerCta && 4 * ne <= (unsigned long long)rk::kMaxRowsPerCta &&
           3 * nc <= (unsigned long long)rk::kMaxRowsPerCta && nv <= (unsigned long long)rk::kMaxRowsPerCta;
}

// A grid of `grid` CTAs in clusters of `cluster`: divisibility, slice capacities, and - the CTAs wait for each
// other's words - that the device can hold all of them at once.
int check_grid(M *m, int grid, int cluster) {
    if (cluster != 1 && cluster != 2 && cluster != 4) return fail(1, "cluster must be 1, 2 or 4");
    if (grid < cluster || grid > m->sms || grid % cluster != 0)
        return fail(1, "grid=%d must be a multiple of cluster=%d and at most %d (the SM count)", grid, cluster, m->sms);
    if (!grid_fits(m->E, (unsigned long long)m->p.Er, (unsigned long long)m->p.Vr, grid))
        return fail(5, "a grid of %d CTAs does not fit n_embed=%llu", grid, m->E);
    if (cluster > 1) {
        cudaLaunchConfig_t cfg{};
        cudaLaunchAttribute attrs[2];
        fill_launch(grid, cluster, m->smem, cfg, attrs, m->stream);
        const bool full = m->E == (unsigned long long)m->cpl * 512ull;
        int nclusters = 0;
        CK(cudaOccupancyMaxActiveClusters(&nclusters, token_entry(m->cpl, full, m->p.trace != nullptr), &cfg));
        if (nclusters * cluster < grid)
            return fail(5, "the device holds %d clusters of %d CTAs at once; a grid of %d needs %d", nclusters, cluster, grid, grid / cluster);
    }
    return 0;
}

int do_load(M *m, const char *path, int quiet) {
    FileReader fr;
    fr.fd = open(path, O_RDONLY);
    if (fr.fd < 0) return fail(2, "Error opening file %s", path);
    int64_t hdr[2];
    int rc = read_exact(fr.fd, hdr, sizeof(hdr), 0);
    if (rc) return rc;
    m->L = (unsigned long long)hdr[0];
    m->E = (unsigned long long)hdr[1];
    const unsigned long long L = m->L, E = m->E, G = (unsigned long long)m->tp_size;
    if (!quiet) {
        printf("n_layers: %llu\nn_embed: %llu\n", L, E);
        fflush(stdout);
    }
    if (L == 0 || L > 4096 || E == 0 || E % 16 != 0 || E > 5120)
        return fail(5, "unsupported model shape: n_layers=%llu n_embed=%llu (need n_embed %% 16 == 0, <= 5120)", L, E);
    if (E % (16 * G) != 0)
        return fail(7, "tensor parallelism: n_embed=%llu is not a multiple of 16 x %llu ranks", E, G);
    struct stat st;
    if (fstat(fr.fd, &st) != 0 || (uint64_t)st.st_size < binfmt::file_bytes(L, E))
        return fail(4, "model file too short: %lld bytes, need %llu", (long long)st.st_size,
                    (unsigned long long)binfmt::file_bytes(L, E));

    CK(cudaSetDevice(m->device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, m->device));
    if (prop.major < 10) return fail(6, "device %d is sm_%d%d; this engine is built for sm_100a only", m->device, prop.major, prop.minor);
    m->sms = prop.multiProcessorCount;
    m->grid = m->sms;
    CK(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
    {
        int coop = 0;
        CK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, m->device));
        if (!coop) return fail(6, "device does not support cooperative launch");
    }

    const unsigned long long Er = E / G;
    const unsigned long long V = binfmt::kVocab;
    const unsigned long long v_lo = V * (unsigned long long)m->tp_rank / G, v_hi = V * ((unsigned long long)m->tp_rank + 1) / G;
    const unsigned long long Vr = v_hi - v_lo;
    m->cpl = chunks_per_lane(E);
    rk::Params &p = m->p;
    p.L = (int)L;
    p.E = (int)E;
    p.G = (int)G;
    p.rank = m->tp_rank;
    p.Er = (int)Er;
    p.Vr = (int)Vr;
    p.vbase = (int)v_lo;
    p.plane_cap = (int)(12 * E);
    p.timeout_ms = G > 1 ? 60000u : 4000u;
    configure_ring(m);
    p.window = std::min(p.stages, 2);
    p.poll_first = 2;
    p.pf_dist = 4;
    p.bwindow = 1;
    p.vseg = G >= 4 ? 1 : G >= 2 ? 2 : 4; // 4E/G bytes per ffn-V row in segments of at most E bytes
    p.cluster = 1;
    if (p.stages < 2) return fail(5, "n_embed=%llu leaves no room for a two-stage ring", E);
    if (!grid_fits(E, Er, Vr, m->grid)) return fail(5, "a grid of %d CTAs does not fit n_embed=%llu", m->grid, E);
    const bool full = E == (unsigned long long)m->cpl * 512ull;
    for (int tr = 0; tr < 3; ++tr) {
        const void *fn = token_entry(m->cpl, full, tr == 1, tr == 2);
        if (!fn) return fail(3, "no kernel for %d chunks per lane", m->cpl);
        CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, rk::kSmemLimit));
    }

    fr.pin_bytes = 64u << 20;
    CK(cudaMallocHost((void **)&fr.pin, fr.pin_bytes));

    // The reference prints every tensor in file order (rwkv.cu:679); keep that UX.
    if (!quiet) {
        for (int t = 0; t < binfmt::kNumTensors; ++t) printf("loading: %s\n", binfmt::name(t));
        fflush(stdout);
    }

    // ---- small parameter tensors, reference dtype and shape (replicated on every rank) ----------
    float *emb, *kr, *vr, *rr, *o1, *o2, *o3, *aor, *aoo, *fkr, *fvr, *frr, *fko, *fvo, *fro, *hr, *ho;
    double *ln, *mixk, *mixv, *mixr, *fmk, *fmr, *decay, *bonus;
#define UP(tid, var)                                                                               \
    if ((rc = upload_tensor(m, fr, tid, &var))) return rc;                                          \
    m->tensors[tid] = var;
    UP(EMBED, emb) UP(LAYERNORMS, ln) UP(MIXK, mixk) UP(MIXV, mixv) UP(MIXR, mixr)
    UP(KR, kr) UP(VR, vr) UP(RR, rr) UP(O1, o1) UP(O2, o2) UP(O3, o3)
    UP(ATTOUTR, aor) UP(ATTOUTO, aoo) UP(FFNMIXK, fmk) UP(FFNMIXV, fmr)
    UP(FFNKR, fkr) UP(FFNVR, fvr) UP(FFNRR, frr) UP(FFNKO, fko) UP(FFNVO, fvo) UP(FFNRO, fro)
    UP(DECAY, decay) UP(BONUS, bonus) UP(HEADR, hr) UP(HEADO, ho)
#undef UP
    p.emb = emb; p.ln = ln; p.mixk = mixk; p.mixv = mixv; p.mixr = mixr; p.fmixk = fmk; p.fmixr = fmr;
    p.decay = decay; p.bonus = bonus;
    p.rk = kr; p.rv = vr; p.rr = rr; p.ro = aor; p.rfk = fkr; p.rfv = fvr; p.rfr = frr; p.rhead = hr;
    {
        double *ed = nullptr;
        if ((rc = dmalloc(m, &ed, (size_t)(L * E)))) return rc;
        rk::k_exp_table<<<(unsigned)((L * E + 255) / 256), 256, 0, m->stream>>>(decay, ed, (size_t)(L * E));
        CK(cudaGetLastError());
        p.expdecay = ed;
    }
    {
        std::vector<double> one(E, 1.0);
        double *d1 = nullptr;
        if ((rc = dmalloc(m, &d1, (size_t)E))) return rc;
        CK(cudaMemcpyAsync(d1, one.data(), E * sizeof(double), cudaMemcpyHostToDevice, m->stream));
        CK(cudaStreamSynchronize(m->stream));
        p.ones = d1;
    }
    if ((rc = centre(m, kr, o1, L * E, &p.ock))) return rc;
    if ((rc = centre(m, vr, o2, L * E, &p.ocv))) return rc;
    if ((rc = centre(m, rr, o3, L * E, &p.ocr))) return rc;
    if ((rc = centre(m, aor, aoo, L * E, &p.oco))) return rc;
    if ((rc = centre(m, fkr, fko, L * E, &p.ocfk))) return rc;
    if ((rc = centre(m, fvr, fvo, L * 4 * E, &p.ocfv))) return rc;
    if ((rc = centre(m, frr, fro, L * E, &p.ocfr))) return rc;
    if ((rc = centre(m, hr, ho, E, &p.ochead))) return rc;

    // ---- uint8 matrices: this rank's slices; stage raw, transpose + centre on the device ----------
    uint8_t *d_raw = nullptr;
    const size_t raw_bytes = std::max<size_t>(4 * Er * E, Vr * E);
    CK(cudaMalloc((void **)&d_raw, raw_bytes));
    const size_t c0 = (size_t)m->tp_rank * Er; // first channel of this rank
    int8_t *wk, *wv, *wr, *wo, *wfk, *wfv, *wfr, *whead;
    rc = upload_matrix(m, fr, KM, L, E, E, 0, E, c0, Er, d_raw, &wk);                         // column split
    if (!rc) rc = upload_matrix(m, fr, VM, L, E, E, 0, E, c0, Er, d_raw, &wv);
    if (!rc) rc = upload_matrix(m, fr, RM, L, E, E, 0, E, c0, Er, d_raw, &wr);
    if (!rc) rc = upload_matrix(m, fr, ATTOUT, L, E, E, c0, Er, 0, E, d_raw, &wo);             // row split
    if (!rc) rc = upload_matrix(m, fr, FFNK, L, E, 4 * E, 0, E, 4 * c0, 4 * Er, d_raw, &wfk);  // column split
    if (!rc) rc = upload_matrix(m, fr, FFNV, L, 4 * E, E, 4 * c0, 4 * Er, 0, E, d_raw, &wfv);  // row split
    if (!rc) rc = upload_matrix(m, fr, FFNR, L, E, E, 0, E, c0, Er, d_raw, &wfr);              // column split
    if (!rc) rc = upload_matrix(m, fr, HEAD, 1, E, V, 0, E, v_lo, Vr, d_raw, &whead);          // column split
    cudaFree(d_raw);
    if (rc) return rc;
    p.wk = wk; p.wv = wv; p.wr = wr; p.wo = wo; p.wfk = wfk; p.wfv = wfv; p.wfr = wfr; p.whead = whead;
    m->tensors[KM] = wk; m->tensors[VM] = wv; m->tensors[RM] = wr; m->tensors[ATTOUT] = wo;
    m->tensors[FFNK] = wfk; m->tensors[FFNV] = wfv; m->tensors[FFNR] = wfr; m->tensors[HEAD] = whead;

    // ---- state, activations, control ------------------------------------------------------------
    const size_t sn = (size_t)(L * E * m->max_gpt);
    if ((rc = dmalloc(m, &p.sxy, sn)) || (rc = dmalloc(m, &p.sdd, sn)) || (rc = dmalloc(m, &m->spp, sn))) return rc;
    for (double *s : {p.sxy, p.sdd, m->spp}) CK(cudaMemsetAsync(s, 0, sn * sizeof(double), m->stream));
    double *b1, *fkb, *fvb;
    float *b3, *b4, *frb;
    if ((rc = dmalloc(m, &p.x, E)) || (rc = dmalloc(m, &p.ctrl, 1)) || (rc = dmalloc(m, &b1, E)) || (rc = dmalloc(m, &fkb, E)) ||
        (rc = dmalloc(m, &fvb, E)) || (rc = dmalloc(m, &b3, E)) || (rc = dmalloc(m, &b4, E)) || (rc = dmalloc(m, &frb, 4 * E)))
        return rc;
    CK(cudaMemsetAsync(p.ctrl, 0, sizeof(rk::Ctrl), m->stream));
    CK(cudaMemsetAsync(p.x, 0, E * sizeof(double), m->stream));
    // exchange block: one allocation, same layout on every rank (exchange.cuh)
    {
        size_t off = 256;
        auto take = [&](size_t bytes) {
            const size_t o = off;
            off = (off + bytes + 255) & ~(size_t)255;
            return o;
        };
        const size_t nb = (size_t)m->grid;
        for (int i = 0; i < 2; ++i) p.off_stat[i] = (unsigned int)take(rk::kRep * 2 * nb * sizeof(rk::TaggedDouble));
        for (int i = 0; i < 5; ++i) p.off_off[i] = (unsigned int)take(rk::kRep * 3 * nb * sizeof(rk::TaggedDouble));
        for (int i = 0; i < 5; ++i) p.off_max[i] = (unsigned int)take(rk::kRep * 3 * nb * 8);
        const size_t vlen[5] = {3 * E, Er, 2 * E, 4 * Er, E};
        for (int i = 0; i < 5; ++i) p.off_vec[i] = (unsigned int)take(vlen[i] * 4);
        for (int i = 0; i < 2; ++i) p.off_in[i] = (unsigned int)take(G * E * sizeof(rk::TaggedDouble));
        p.off_sr = (unsigned int)take(E * 8);
        p.off_arg = (unsigned int)take(G * nb * sizeof(rk::TaggedDouble));
        p.off_done = (unsigned int)take(G * nb * 8);
        p.off_smp = (unsigned int)take(rk::kRep * 3 * nb * sizeof(rk::TaggedDouble));
        p.off_logits = (unsigned int)take(V * 4);
        p.off_saa = take(sn * 8);
        p.off_sbb = take(sn * 8);
        m->xch_bytes = off;
        unsigned char *x = nullptr;
        if ((rc = dmalloc(m, &x, m->xch_bytes))) return rc;
        CK(cudaMemsetAsync(x, 0, m->xch_bytes, m->stream));
        for (int g = 0; g < rk::kMaxRanks; ++g) p.xch[g] = x; // peers are wired by rwkv_b200_tp_import
    }
    float *logits = reinterpret_cast<float *>(p.xch[0] + p.off_logits);
    double *saa = reinterpret_cast<double *>(p.xch[0] + p.off_saa), *sbb = reinterpret_cast<double *>(p.xch[0] + p.off_sbb);
    m->tensors[X] = p.x;
    m->tensors[STATEXY] = p.sxy; m->tensors[STATEAA] = saa; m->tensors[STATEBB] = sbb;
    m->tensors[STATEPP] = m->spp; m->tensors[STATEDD] = p.sdd;
    m->tensors[BUFFER1] = b1; m->tensors[BUFFER2] = logits; m->tensors[BUFFER3] = b3; m->tensors[BUFFER4] = b4;
    m->tensors[FFNKBUFFER] = fkb; m->tensors[FFNVBUFFER] = fvb; m->tensors[FFNRBUFFER] = frb;

    CK(cudaMallocHost((void **)&m->h_ctrl, sizeof(rk::Ctrl) * m->max_gpt));
    CK(cudaMallocHost((void **)&m->h_logits, sizeof(float) * V * m->max_gpt));
    CK(cudaMallocHost((void **)&m->h_next, sizeof(unsigned long long)));
    CK(cudaHostAlloc((void **)&m->h_diag, sizeof(rk::Diag), cudaHostAllocMapped));
    memset(m->h_diag, 0, sizeof(rk::Diag));
    CK(cudaHostGetDevicePointer((void **)&p.diag, m->h_diag, 0));
    memset(m->h_logits, 0, sizeof(float) * V * m->max_gpt);
    CK(cudaStreamSynchronize(m->stream));
    return 0;
}

int check_model(const M *m) {
    if (!m) return fail(1, "null model handle");
    return 0;
}

float *dev_logits(M *m) { return reinterpret_cast<float *>(m->p.xch[m->tp_rank] + m->p.off_logits); }

} // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

const char *rwkv_b200_last_error(void) { return g_err.c_str(); }
int rwkv_b200_abi_version(void) { return 2; }

int rwkv_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int rwkv_b200_load_tp(const char *path, unsigned long long max_gpt, int device, int quiet, int tp_rank, int tp_size,
                      rwkv_b200_model **out, unsigned long long *n_layers, unsigned long long *n_embed) {
    if (!path || !out) return fail(1, "null argument");
    *out = nullptr;
    if (tp_size < 1 || tp_size > rk::kMaxRanks || tp_rank < 0 || tp_rank >= tp_size)
        return fail(7, "tensor parallelism: rank %d of %d is not supported (1..8 ranks)", tp_rank, tp_size);
    if (rwkv_b200_device_count() <= device || device < 0)
        return fail(6, "CUDA device %d not available (no CPU fallback exists)", device);
    M *m = new M;
    m->device = device;
    m->max_gpt = max_gpt ? max_gpt : 1;
    m->tp_rank = tp_rank;
    m->tp_size = tp_size;
    int rc = do_load(m, path, quiet);
    if (rc) {
        std::string keep = g_err;
        rwkv_b200_free(m);
        g_err = keep;
        return rc;
    }
    *out = m;
    if (n_layers) *n_layers = m->L;
    if (n_embed) *n_embed = m->E;
    return 0;
}

int rwkv_b200_load(const char *path, unsigned long long max_gpt, int device, int quiet, rwkv_b200_model **out,
                   unsigned long long *n_layers, unsigned long long *n_embed) {
    return rwkv_b200_load_tp(path, max_gpt, device, quiet, 0, 1, out, n_layers, n_embed);
}

void rwkv_b200_free(rwkv_b200_model *m) {
    if (!m) return;
    cudaSetDevice(m->device);
    if (m->stream) cudaStreamSynchronize(m->stream);
    rk::prefill_free(m->pf);
    for (void *p : m->ipc_opened) cudaIpcCloseMemHandle(p);
    for (void *p : m->allocs) cudaFree(p);
    if (m->h_ctrl) cudaFreeHost(m->h_ctrl);
    if (m->h_logits) cudaFreeHost(m->h_logits);
    if (m->h_next) cudaFreeHost(m->h_next);
    if (m->h_sample) cudaFreeHost(m->h_sample);
    if (m->d_gen) cudaFree(m->d_gen);
    if (m->h_gen) cudaFreeHost(m->h_gen);
    if (m->h_diag) cudaFreeHost(m->h_diag);
    if (m->stream) cudaStreamDestroy(m->stream);
    cudaGetLastError(); // a context killed by a trap makes every call above fail; do not leave that as "last error"
    delete m;
}

void *rwkv_b200_tensor(rwkv_b200_model *m, int index) {
    if (!m || index < 0 || index >= RWKV_B200_NUM_TENSORS) return nullptr;
    return m->tensors[index];
}
unsigned long long rwkv_b200_n_layers(const rwkv_b200_model *m) { return m ? m->L : 0; }
unsigned long long rwkv_b200_n_embed(const rwkv_b200_model *m) { return m ? m->E : 0; }
unsigned long long rwkv_b200_max_gpt(const rwkv_b200_model *m) { return m ? m->max_gpt : 0; }

void *rwkv_b200_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (bytes == 0) bytes = 1;
    if (cudaMallocHost(&p, bytes) == cudaSuccess) return p;
    cudaGetLastError();
    // No driver (tokenizer-only use): tag the block so host_free knows it came from malloc.
    uint64_t *raw = (uint64_t *)malloc(bytes + 16);
    if (!raw) return nullptr;
    raw[0] = 0x6d616c6c6f636564ULL;
    return raw + 2;
}
void rwkv_b200_host_free(void *p) {
    if (!p) return;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) == cudaSuccess && a.type == cudaMemoryTypeHost) {
        cudaFreeHost(p);
        return;
    }
    cudaGetLastError();
    uint64_t *raw = (uint64_t *)p - 2;
    if (raw[0] == 0x6d616c6c6f636564ULL) free(raw);
}

int rwkv_b200_state_upload(rwkv_b200_model *m, const double *xy, const double *aa, const double *bb,
                           const double *pp, const double *dd, unsigned long long slots) {
    int rc = check_model(m);
    if (rc) return rc;
    if (slots > m->max_gpt) return fail(1, "state_upload: %llu slots > max_gpt %llu", slots, m->max_gpt);
    CK(cudaSetDevice(m->device));
    const size_t n = (size_t)(m->L * m->E * slots) * sizeof(double);
    const double *src[5] = {xy, aa, bb, pp, dd};
    double *dst[5] = {m->p.sxy, (double *)m->tensors[STATEAA], (double *)m->tensors[STATEBB], m->spp, m->p.sdd};
    for (int i = 0; i < 5; ++i)
        if (src[i]) CK(cudaMemcpyAsync(dst[i], src[i], n, cudaMemcpyHostToDevice, m->stream));
    SYNC(m);
    return 0;
}

int rwkv_b200_state_download(rwkv_b200_model *m, double *xy, double *aa, double *bb, double *pp, double *dd,
                             unsigned long long slots) {
    int rc = check_model(m);
    if (rc) return rc;
    if (slots > m->max_gpt) return fail(1, "state_download: %llu slots > max_gpt %llu", slots, m->max_gpt);
    CK(cudaSetDevice(m->device));
    const size_t n = (size_t)(m->L * m->E * slots) * sizeof(double);
    double *dst[5] = {xy, aa, bb, pp, dd};
    const double *src[5] = {m->p.sxy, (double *)m->tensors[STATEAA], (double *)m->tensors[STATEBB], m->spp, m->p.sdd};
    for (int i = 0; i < 5; ++i)
        if (dst[i]) CK(cudaMemcpyAsync(dst[i], src[i], n, cudaMemcpyDeviceToHost, m->stream));
    SYNC(m);
    return 0;
}

int rwkv_b200_state_zero(rwkv_b200_model *m) {
    int rc = check_model(m);
    if (rc) return rc;
    CK(cudaSetDevice(m->device));
    const size_t n = (size_t)(m->L * m->E * m->max_gpt) * sizeof(double);
    for (double *s : {m->p.sxy, (double *)m->tensors[STATEAA], (double *)m->tensors[STATEBB], m->p.sdd, m->spp})
        CK(cudaMemsetAsync(s, 0, n, m->stream));
    SYNC(m);
    return 0;
}

int rwkv_b200_forward(rwkv_b200_model *m, const unsigned long long *tokens, unsigned long long n_tokens, int mode,
                      float *logits_out) {
    int rc = check_model(m);
    if (rc) return rc;
    if (!tokens || n_tokens == 0) return fail(1, "forward: no tokens");
    if (n_tokens > m->max_gpt) return fail(1, "Context too large, max context is %llu", m->max_gpt);
    CK(cudaSetDevice(m->device));
    const size_t V = binfmt::kVocab;
    for (unsigned long long t = 0; t < n_tokens; ++t)
        if (tokens[t] >= V) return fail(1, "token id %llu out of range", tokens[t]);
    if (n_tokens >= (unsigned long long)m->pf.min_tokens && m->tp_size == 1 && rk::prefill_enabled(m->pf)) {
        rc = rk::prefill_forward(m->pf, m->p, m->stream, tokens, (int)n_tokens, mode == RWKV_B200_MODE_PARRALEL,
                                 logits_out ? m->h_logits : nullptr);
        if (rc) return fail(rc, "%s", rk::prefill_error());
        m->launches += rk::prefill_launches(m->pf);
        SYNC(m);
        if (logits_out && logits_out != m->h_logits) memcpy(logits_out, m->h_logits, n_tokens * V * sizeof(float));
        return 0;
    }
    for (unsigned long long t = 0; t < n_tokens; ++t) {
        rk::Ctrl &c = m->h_ctrl[t];
        c.token = tokens[t];
        c.next = 0;
        c.slot = (mode == RWKV_B200_MODE_PARRALEL) ? t : 0;
        c.pos = 0;
        CK(cudaMemcpyAsync(m->p.ctrl, &c, sizeof(rk::Ctrl), cudaMemcpyHostToDevice, m->stream));
        if ((rc = launch_token(m, 0, false, nullptr, m->stream))) return rc;
        if (logits_out)
            CK(cudaMemcpyAsync(m->h_logits + t * V, dev_logits(m), V * sizeof(float), cudaMemcpyDeviceToHost, m->stream));
    }
    SYNC(m);
    if (logits_out && logits_out != m->h_logits) memcpy(logits_out, m->h_logits, n_tokens * V * sizeof(float));
    return 0;
}

int rwkv_b200_forward_greedy(rwkv_b200_model *m, unsigned long long token, unsigned long long *next, float *logits_out) {
    int rc = check_model(m);
    if (rc) return rc;
    const size_t V = binfmt::kVocab;
    if (token >= V) return fail(1, "token id %llu out of range", token);
    CK(cudaSetDevice(m->device));
    rk::Ctrl &c = m->h_ctrl[0];
    c.token = token;
    c.next = 0;
    c.slot = 0;
    c.pos = 0;
    CK(cudaMemcpyAsync(m->p.ctrl, &c, sizeof(rk::Ctrl), cudaMemcpyHostToDevice, m->stream));
    if ((rc = launch_token(m, 0, true, nullptr, m->stream))) return rc;
    CK(cudaMemcpyAsync(m->h_next, &m->p.ctrl->next, sizeof(unsigned long long), cudaMemcpyDeviceToHost, m->stream));
    if (logits_out) CK(cudaMemcpyAsync(m->h_logits, dev_logits(m), V * sizeof(float), cudaMemcpyDeviceToHost, m->stream));
    SYNC(m);
    if (next) *next = *m->h_next;
    if (logits_out && logits_out != m->h_logits) memcpy(logits_out, m->h_logits, V * sizeof(float));
    return 0;
}

float *rwkv_b200_logits_host(rwkv_b200_model *m) { return m ? m->h_logits : nullptr; }

int rwkv_b200_sample_typical(rwkv_b200_model *m, float temp, double u, unsigned long long *token, double *margin) {
    int rc = check_model(m);
    if (rc) return rc;
    if (!token) return fail(1, "null argument");
    CK(cudaSetDevice(m->device));
    if (!m->d_sample) {
        if ((rc = dmalloc(m, &m->d_sample, 2))) return rc;
        CK(cudaMallocHost((void **)&m->h_sample, 2 * sizeof(double)));
    }
    // the reference applies the temperature as probs ^ uint8(1 / temp) (include/rwkv/sampler/typical.h)
    const int exponent = temp != 1.0f ? (int)(unsigned char)(1.0 / (double)temp) : 1;
    rk::k_sample_typical<<<1, rk::kSampleThreads, 0, m->stream>>>(dev_logits(m), (int)binfmt::kVocab, exponent, u, m->d_sample);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(m->h_sample, m->d_sample, 2 * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
    SYNC(m);
    *token = (unsigned long long)m->h_sample[0];
    if (margin) *margin = m->h_sample[1];
    m->launches += 1;
    return 0;
}

int rwkv_b200_generate(rwkv_b200_model *m, unsigned long long first_token, unsigned long long n, int how, float temp,
                       const double *uniforms, const unsigned long long *stop, int n_stop, unsigned long long *tokens_out,
                       unsigned long long *n_out, float *logits_out) {
    int rc = check_model(m);
    if (rc) return rc;
    const unsigned long long V = binfmt::kVocab;
    if (how != RWKV_B200_GEN_GREEDY && how != RWKV_B200_GEN_TYPICAL) return fail(1, "generate: `how` must be GREEDY (0) or TYPICAL (1)");
    if (n == 0 || !tokens_out || !n_out) return fail(1, "generate: n must be positive and tokens_out, n_out non-null");
    *n_out = 0;
    if (m->tp_size > 1) return fail(7, "generate: not supported with tensor parallelism (%d ranks)", m->tp_size);
    if (first_token >= V) return fail(1, "generate: token id %llu out of range", first_token);
    if (n_stop < 0 || n_stop > rk::kMaxStop || (n_stop > 0 && !stop)) return fail(1, "generate: 0..%d stop ids", rk::kMaxStop);
    for (int k = 0; k < n_stop; ++k)
        if (stop[k] >= V) return fail(1, "generate: stop id %llu out of range", stop[k]);
    const bool typ = how == RWKV_B200_GEN_TYPICAL;
    int exponent = 1;
    if (typ) {
        if (!uniforms) return fail(1, "generate: TYPICAL needs n uniforms");
        for (unsigned long long i = 0; i < n; ++i)
            if (!(uniforms[i] >= 0.0 && uniforms[i] < 1.0)) return fail(1, "generate: uniform %llu = %.17g is outside [0, 1)", i, uniforms[i]);
        // uint8(1 / temp) as include/rwkv/sampler/typical.h computes it; defined for 1 / temp < 256
        if (!(temp > 1.0f / 256.0f)) return fail(1, "generate: temp must be > 1/256 (got %g)", (double)temp);
        exponent = temp != 1.0f ? (int)(uint8_t)(1.0 / (double)temp) : 1;
    }
    CK(cudaSetDevice(m->device));
    if (m->gen_cap < n) {
        if (m->d_gen) cudaFree(m->d_gen);
        if (m->h_gen) cudaFreeHost(m->h_gen);
        m->d_gen = m->h_gen = nullptr;
        m->gen_cap = 0;
        CK(cudaMalloc((void **)&m->d_gen, 24 * n));
        CK(cudaMallocHost((void **)&m->h_gen, 24 * n));
        m->gen_cap = n;
    }
    const unsigned long long cap = m->gen_cap;
    double *d_u = reinterpret_cast<double *>(m->d_gen), *h_u = reinterpret_cast<double *>(m->h_gen);
    unsigned long long *d_t = reinterpret_cast<unsigned long long *>(m->d_gen + 8 * cap), *h_t = reinterpret_cast<unsigned long long *>(m->h_gen + 8 * cap);
    double *d_mg = reinterpret_cast<double *>(m->d_gen + 16 * cap), *h_mg = reinterpret_cast<double *>(m->h_gen + 16 * cap);
    if (typ) {
        memcpy(h_u, uniforms, n * sizeof(double));
        CK(cudaMemcpyAsync(d_u, h_u, n * sizeof(double), cudaMemcpyHostToDevice, m->stream));
    }
    rk::Params &p = m->p;
    p.exponent = exponent;
    p.n_stop = n_stop;
    for (int k = 0; k < rk::kMaxStop; ++k) p.stop[k] = k < n_stop ? stop[k] : 0;
    p.margin_min = m->sample_margin;
    p.uniforms = d_u;
    p.gen_tokens = d_t;
    p.gen_margins = d_mg;
    auto is_stop = [&](unsigned long long t) { return std::find(stop, stop + n_stop, t) != stop + n_stop; };
    // exchange epochs after each enqueued launch: launches that exited at entry must not keep theirs (DESIGN 4.1)
    std::vector<std::pair<unsigned int, unsigned int>> ep(n + 1);
    std::vector<float> fallback_logits;
    unsigned long long done = 0, tok = first_token;
    // The first segment enqueues every step (no halt: one synchronisation per call). After a halt the launches behind
    // it exited at entry; the next segment enqueues at most twice what the last one ran + 16, so frequent halts
    // (sample_margin near 1, or logits out of the host's range every step) cost O(n) launches, not O(n^2).
    unsigned long long chunk = n;
    for (;;) {
        rk::Ctrl &c = m->h_ctrl[0];
        c = rk::Ctrl{0, tok, 0, done, 0};
        CK(cudaMemcpyAsync(p.ctrl, &c, sizeof(rk::Ctrl), cudaMemcpyHostToDevice, m->stream));
        const unsigned long long todo = std::min(n - done, chunk);
        ep[0] = {m->epoch, m->tk};
        for (unsigned long long i = 0; i < todo; ++i) {
            if ((rc = launch_token(m, 1, !typ, nullptr, m->stream, true))) return rc;
            ep[i + 1] = {m->epoch, m->tk};
        }
        CK(cudaMemcpyAsync(&c, p.ctrl, sizeof(rk::Ctrl), cudaMemcpyDeviceToHost, m->stream));
        CK(cudaMemcpyAsync(h_t + done, d_t + done, todo * sizeof(unsigned long long), cudaMemcpyDeviceToHost, m->stream));
        if (typ) CK(cudaMemcpyAsync(h_mg + done, d_mg + done, todo * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
        if (logits_out) CK(cudaMemcpyAsync(m->h_logits, dev_logits(m), V * sizeof(float), cudaMemcpyDeviceToHost, m->stream));
        SYNC(m);
        const unsigned long long ran = c.pos - done;
        if (ran == 0 || ran > todo || (ran < todo && !c.halt))
            return fail(8, "generate: the device ran %llu of %llu steps (halt %llu)", ran, todo, c.halt);
        m->epoch = ep[ran].first;
        m->tk = ep[ran].second;
        done = c.pos;
        const unsigned long long s = done - 1;
        if (!c.halt) {
            if (done == n) break;
            tok = h_t[s]; // a bounded segment ran to its end
            continue;
        }
        chunk = 2 * ran + 16;
        if (typ && (!(h_mg[s] >= m->sample_margin) || h_mg[s] < 0.0)) {
            // u too close to a boundary for the device's sums (or outside their range): the host's arithmetic decides
            const float *lg = m->h_logits;
            if (!logits_out) {
                fallback_logits.resize(V);
                CK(cudaMemcpy(fallback_logits.data(), dev_logits(m), V * sizeof(float), cudaMemcpyDeviceToHost));
                lg = fallback_logits.data();
            }
            h_t[s] = (unsigned long long)typical_with_u(lg, temp, uniforms[s]);
        }
        tok = h_t[s];
        if (done == n || is_stop(tok)) break;
    }
    memcpy(tokens_out, h_t, done * sizeof(unsigned long long));
    *n_out = done;
    if (logits_out && logits_out != m->h_logits) memcpy(logits_out, m->h_logits, V * sizeof(float));
    return 0;
}

int rwkv_b200_decode_timed(rwkv_b200_model *m, const unsigned long long *tokens, unsigned long long n,
                           int teacher_forced, float *ms) {
    int rc = check_model(m);
    if (rc) return rc;
    if (!tokens || n == 0 || !ms) return fail(1, "decode_timed: bad arguments");
    CK(cudaSetDevice(m->device));
    const unsigned long long cnt = teacher_forced ? n : 1;
    for (unsigned long long i = 0; i < cnt; ++i)
        if (tokens[i] >= binfmt::kVocab) return fail(1, "token id %llu out of range", tokens[i]);
    unsigned long long *d_tok = nullptr;
    cudaEvent_t a = nullptr, b = nullptr;
    cudaError_t e = cudaMalloc((void **)&d_tok, cnt * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemcpy(d_tok, tokens, cnt * sizeof(unsigned long long), cudaMemcpyHostToDevice);
    rk::Ctrl c{tokens[0], tokens[0], 0, 0};
    if (e == cudaSuccess) e = cudaStreamSynchronize(m->stream);
    if (e == cudaSuccess) e = cudaMemcpy(m->p.ctrl, &c, sizeof(rk::Ctrl), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaEventCreate(&a);
    if (e == cudaSuccess) e = cudaEventCreate(&b);
    if (e == cudaSuccess) e = cudaEventRecord(a, m->stream);
    rc = 0;
    for (unsigned long long i = 0; i < n && e == cudaSuccess && rc == 0; ++i)
        rc = launch_token(m, teacher_forced ? 2 : 1, !teacher_forced, d_tok, m->stream);
    if (e == cudaSuccess && rc == 0) e = cudaEventRecord(b, m->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(m->stream);
    if (e == cudaSuccess && rc == 0) e = cudaEventElapsedTime(ms, a, b);
    if (a) cudaEventDestroy(a);
    if (b) cudaEventDestroy(b);
    if (d_tok) cudaFree(d_tok);
    if (rc) return rc;
    if (e != cudaSuccess) return sync_failed(m, e, "decode_timed");
    return 0;
}

int rwkv_b200_kernel_count(void) { return 1; }
const char *rwkv_b200_kernel_name(int k) { return k == 0 ? kKernelNames[0] : ""; }

int rwkv_b200_profile(rwkv_b200_model *m, const unsigned long long *tokens, unsigned long long n, float *ms_sum,
                      unsigned long long *launches, double *bytes) {
    int rc = check_model(m);
    if (rc) return rc;
    if (!tokens || !ms_sum || !launches || !bytes) return fail(1, "profile: bad arguments");
    CK(cudaSetDevice(m->device));
    ms_sum[0] = 0.f;
    launches[0] = 0;
    // algorithmic HBM bytes of one launch on this rank: its share of the weights + the vectors
    const double E = (double)m->E, V = (double)binfmt::kVocab, L = (double)m->L, G = (double)m->tp_size;
    bytes[0] = (13.0 * L * E * E + V * E) / G + ((double)binfmt::algorithmic_bytes_per_token(m->L, m->E) - (13.0 * L * E * E + V * E));
    cudaEvent_t a = nullptr, b = nullptr;
    CK(cudaEventCreate(&a));
    cudaError_t e = cudaEventCreate(&b);
    rc = 0;
    for (unsigned long long t = 0; t < n && e == cudaSuccess && rc == 0; ++t) {
        if (tokens[t] >= binfmt::kVocab) {
            rc = fail(1, "token id out of range");
            break;
        }
        rk::Ctrl c{tokens[t], 0, 0, 0};
        e = cudaMemcpyAsync(m->p.ctrl, &c, sizeof(rk::Ctrl), cudaMemcpyHostToDevice, m->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(m->stream);
        if (e == cudaSuccess) e = cudaEventRecord(a, m->stream);
        if (e == cudaSuccess) rc = launch_token(m, 0, true, nullptr, m->stream);
        if (e == cudaSuccess && rc == 0) e = cudaEventRecord(b, m->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(m->stream);
        float t_ms = 0.f;
        if (e == cudaSuccess && rc == 0) e = cudaEventElapsedTime(&t_ms, a, b);
        ms_sum[0] += t_ms;
        launches[0] += 1;
    }
    cudaEventDestroy(a);
    if (b) cudaEventDestroy(b);
    if (rc) return rc;
    if (e != cudaSuccess) return sync_failed(m, e, "profile");
    return 0;
}

unsigned long long rwkv_b200_launch_count(const rwkv_b200_model *m) { return m ? m->launches : 0; }

int rwkv_b200_set_option(rwkv_b200_model *m, const char *key, const char *value) {
    int rc = check_model(m);
    if (rc) return rc;
    if (!key || !value) return fail(1, "set_option: null");
    const std::string k = key;
    const int v = atoi(value);
    if (k == "trace") {
        if (v && !m->p.trace) {
            unsigned long long *t = nullptr;
            if (dmalloc(m, &t, (size_t)rk::kMaxGrid * rk::kTraceMax)) return fail(1, "trace alloc failed");
            cudaMemset(t, 0, (size_t)rk::kMaxGrid * rk::kTraceMax * 8);
            m->p.trace = t;
            unsigned long long *pt = nullptr;
            if (dmalloc(m, &pt, (size_t)2 * rk::kMaxGrid * rk::kTileTraceMax)) return fail(1, "trace alloc failed");
            cudaMemset(pt, 0, (size_t)2 * rk::kMaxGrid * rk::kTileTraceMax * 8);
            m->p.ptrace = pt;
        } else if (!v) {
            m->p.trace = nullptr;
            m->p.ptrace = nullptr;
        }
    } else if (k == "max_layers") m->max_layers = v;
    else if (k == "issue_gap") {
        if (v < 0 || v > 100000) return fail(1, "issue_gap is a cycle count in 0..100000");
        m->p.issue_gap = v;
    } else if (k == "window") {
        if (v < 1 || v > rk::kMaxStages) return fail(1, "window must be 1..%d", rk::kMaxStages);
        m->p.window = v;
    } else if (k == "cluster" || k == "grid") {
        const int c = k == "cluster" ? v : m->p.cluster, g = k == "grid" ? v : m->grid;
        if (int rc2 = check_grid(m, g, c)) return rc2;
        m->p.cluster = c;
        m->grid = g;
    } else if (k == "bwindow") {
        if (v < 1 || v > rk::kMaxStages) return fail(1, "bwindow must be 1..%d", rk::kMaxStages);
        m->p.bwindow = v;
    } else if (k == "pf_dist") {
        if (v < 0 || v > 64) return fail(1, "pf_dist is 0..64 tiles");
        m->p.pf_dist = v;
    } else if (k == "poll_first") {
        if (v < 0 || v > 2) return fail(1, "poll_first is 0, 1 or 2");
        m->p.poll_first = v;
    } else if (k == "dbg") {
        m->p.dbg = v;
    } else if (k == "timeout_ms") {
        if (v < 1) return fail(1, "timeout_ms must be positive");
        m->p.timeout_ms = (unsigned int)v;
    } else if (k == "stages") {
        if (v < 2 || v > rk::kMaxStages) return fail(1, "stages must be 2..%d", rk::kMaxStages);
        const size_t smem = rk::smem_bytes(v, m->p.tile_bytes, m->p.plane_cap);
        if (smem > (size_t)rk::kSmemLimit) return fail(1, "stages=%d needs %zu bytes of shared memory", v, smem);
        m->p.stages = v;
        m->smem = smem;
    } else if (k == "prefill") {
        m->pf.disabled = v == 0;
    } else if (k == "prefill_graph") {
        m->pf.use_graph = v != 0;
    } else if (k == "sample_margin") {
        const double d = atof(value);
        if (!(d >= 0.0 && d <= 1.0)) return fail(1, "sample_margin must be in [0, 1]");
        m->sample_margin = d;
    } else if (k == "prefill_min") {
        if (v < 2) return fail(1, "prefill_min must be >= 2");
        m->pf.min_tokens = v;
    } else return fail(1, "unknown option '%s'", key);
    return 0;
}

// Debug/test hook: copy a named device vector to the host. Returns the element count.
long long rwkv_b200_debug_read(rwkv_b200_model *m, const char *name, void *dst, size_t dst_bytes) {
    if (check_model(m) || !name || !dst) return -1;
    cudaSetDevice(m->device);
    const std::string k = name;
    const void *src = nullptr;
    size_t bytes = 0, count = 0;
    const size_t E = m->E;
    if (k == "x") src = m->p.x, count = E, bytes = E * 8;
    else if (k == "logits") src = dev_logits(m), count = binfmt::kVocab, bytes = 4 * binfmt::kVocab;
    else if (k == "trace" && m->p.trace) src = m->p.trace, count = (size_t)m->grid * rk::kTraceMax, bytes = count * 8;
    else if (k == "ptrace" && m->p.ptrace) src = m->p.ptrace, count = (size_t)2 * m->grid * rk::kTileTraceMax, bytes = count * 8;
    else return -1;
    if (dst_bytes < bytes) return -1;
    if (cudaStreamSynchronize(m->stream) != cudaSuccess) return -1;
    if (cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    return (long long)count;
}

size_t rwkv_b200_tp_buffer_bytes(const rwkv_b200_model *m) { return m ? m->xch_bytes : 0; }

int rwkv_b200_tp_export(rwkv_b200_model *m, void *ipc_handle_64) {
    if (check_model(m) || !ipc_handle_64) return fail(1, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaSetDevice(m->device);
    CK(cudaStreamSynchronize(m->stream)); // the block is zero-filled before anybody maps it
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, m->p.xch[m->tp_rank]));
    memcpy(ipc_handle_64, &h, 64);
    return 0;
}

int rwkv_b200_tp_import(rwkv_b200_model *m, const void *ipc_handles) {
    if (check_model(m) || !ipc_handles) return fail(1, "null argument");
    if (m->tp_wired) return fail(7, "peer exchange blocks already imported");
    cudaSetDevice(m->device);
    const unsigned char *hs = static_cast<const unsigned char *>(ipc_handles);
    for (int g = 0; g < m->tp_size; ++g) {
        if (g == m->tp_rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, hs + 64 * (size_t)g, 64);
        void *ptr = nullptr;
        CK(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
        m->ipc_opened.push_back(ptr);
        m->p.xch[g] = static_cast<unsigned char *>(ptr);
    }
    m->tp_wired = true;
    return 0;
}

} // extern "C"
