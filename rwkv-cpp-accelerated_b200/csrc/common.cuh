// common.cuh — parameters, shared-memory map and PTX helpers of the sm_100a RWKV-v4 uint8 decode path.
//
// The arithmetic idea (why three byte limbs): the reference computes
//   y_k = sum_j x_j * (w_jk * r_j + o_j)                     (include/rwkv/cuda/rwkv.cu:279-294)
// in fp32 with one I2F and two FMAs per weight byte. Factorised as
//   y_k = sum_j (x_j r_j) * w'_jk + sum_j x_j * (128 r_j + o_j),      w' = w - 128 (int8 = byte ^ 0x80)
// the per-byte work is 3/4 of an IDP.4A: the activation vector xs_j = x_j r_j is quantised once per phase
// to a 23-bit integer q_j relative to max|xs| and the three low bytes of q_j are the limbs (two unsigned
// digits, one signed top digit). Accumulation is exact int32, recombination exact int64, so results are
// bit-deterministic and independent of how rows are distributed over CTAs or GPUs.
//
// HBM layout of a matrix: row-major [out][in] int8, so the rows one CTA owns are one contiguous byte
// range -> 1-D bulk TMA copies, no tensor maps.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace rk {

constexpr int kVocab = 50277;
constexpr int kWarps = 8;                  // consumer warps: one per unit of a tile
constexpr int kConsumers = kWarps * 32;    // 256
constexpr int kProducerThreads = 128;      // a whole warpgroup, so that setmaxnreg can move its registers
constexpr int kThreads = kConsumers + kProducerThreads;
constexpr int kProducerRegs = 40;
constexpr int kConsumerRegs = 232;         // 256 x (232 - 168) = 128 x (168 - 40)
constexpr int kMaxStages = 12;
constexpr int kMaxGrid = 160;              // CTAs per rank (one per SM)
constexpr int kMaxRanks = 8;
constexpr int kMaxSlice = 64;              // residual elements / channels one CTA owns
constexpr int kMaxKeys = 160;              // ffn key channels one CTA owns
constexpr int kRep = 8;                    // replicas of the per-CTA exchange records (readers of one L2 line / kRep)
constexpr int kMaxRowsPerCta = 1024;       // res64 capacity (rows x segments of one CTA)
constexpr int kTraceMax = 2048;            // trace stamps per CTA (debug)
constexpr int kTileTraceMax = 4096;        // tiles per CTA recorded by the tile trace (debug)
constexpr int kQMax = 4194303;             // 2^22 - 1: largest |q| of the activation quantiser
constexpr int kSmemLimit = 232448;         // opt-in dynamic shared memory per CTA on sm_100
constexpr int kMaxStop = 8;                // stop ids of a generate run

// Device-resident control block of one model (one per rank).
struct Ctrl {
    unsigned long long token; // input token of the current forward (feed_mode 0)
    unsigned long long next;  // argmax of the last logits (greedy)
    unsigned long long slot;  // state slot (PARRALEL mode)
    unsigned long long pos;   // cursor into a device-resident token stream (feed_mode 2); generate: steps done
    unsigned long long halt;  // generate: nonzero = the next launches exit at entry (stop token or small margin)
};

// Diagnostic record written to mapped host memory just before a timeout trap, so that the host can say
// WHICH wait did not complete (the CUDA context is unusable after __trap()).
struct Diag {
    unsigned int code;     // 0 = nothing; see kDiag*
    unsigned int rank, cta, thread;
    unsigned int layer, kind, expect, seen;
    unsigned long long aux;
};
constexpr unsigned int kDiagStats = 1, kDiagVec = 2, kDiagOff = 3, kDiagPeerSum = 4, kDiagSr = 5, kDiagDone = 6,
                       kDiagArg = 7, kDiagRingFull = 8, kDiagRingEmpty = 9, kDiagPlanesFree = 10, kDiagPlanesReady = 11,
                       kDiagSample = 12;

// Everything the token kernel needs, passed by value (__grid_constant__).
// G ranks (GPUs) decode ONE stream together (G = 1: a single GPU). Split (SURVEY 8e):
//   K, V, R, ffn-R : column split - rank g owns output channels [g*Er, (g+1)*Er), inputs all E
//   out-proj       : row split    - inputs = the rank's channels, outputs all E -> partial sums, exchanged
//   ffn-K          : column split - rank g owns key channels [g*4Er, (g+1)*4Er)
//   ffn-V          : row split    - inputs = the rank's key channels, outputs all E -> partial sums, exchanged
//   head           : column split over the vocabulary
// The residual stream, layernorm and token shift are replicated on every rank (bit-identical).
struct Params {
    int L, E;
    int G, rank;
    int Er;                 // E / G
    int Vr, vbase;          // vocabulary rows of this rank, first global row
    int tile_bytes, stages; // ring: `stages` tiles of 8*E bytes
    int plane_cap;          // bytes reserved for limb planes in shared memory
    int L_run;              // layers to run (debug knob; normally == L)
    int feed_mode;          // 0: ctrl->token, 1: ctrl->next (free-running), 2: stream[ctrl->pos]
    int greedy;             // 1: finish with an on-device argmax into ctrl->next
    int issue_gap;          // minimum SM cycles between two bulk-copy issues of the producer (0 = unpaced)
    int window;             // bulk copies in flight per CTA (<= stages)
    int cluster;            // CTAs per thread-block cluster (1, 2 or 4): they split the gather and write each other's limb planes
    int vseg;               // segments per ffn-V row (4E/G bytes): 4, 2 or 1 so that a segment is <= E bytes and a tile 8 / vseg rows
    int bwindow;            // bulk copies in flight per CTA while the consumers exchange vectors (latency of their loads)
    int pf_dist;            // tiles the L2 prefetch cursor runs ahead of the ring (0 = no L2 prefetch)
    int dbg;                // debug experiments (bit 0: run the slice statistics twice, cold / warm code)
    int poll_first;         // gather: 1 = poll the first 16 bytes before fetching the rest, 0 = fetch everything at once
    unsigned int ep0;       // epoch before this token: layer l tags its exchanges with ep0 + 1 + l
    unsigned int tk;        // token epoch (tags of the once-per-token exchanges)
    unsigned int timeout_ms;
    // this rank's weight shards, int8 row-major
    const int8_t *wk, *wv, *wr;  // [L][Er][E]
    const int8_t *wo;            // [L][E][Er]
    const int8_t *wfr;           // [L][Er][E]
    const int8_t *wfk;           // [L][4Er][E]
    const int8_t *wfv;           // [L][E][4Er]
    const int8_t *whead;         // [Vr][E]
    // per-input-row scale r and centred offset oc = 128*r + o (full vectors on every rank)
    const float *rk, *rv, *rr, *ro, *rfk, *rfv, *rfr, *rhead;
    const float *ock, *ocv, *ocr, *oco, *ocfk, *ocfv, *ocfr, *ochead;
    const double *ln;                                  // [4(L+1)][E]
    const double *mixk, *mixv, *mixr, *fmixk, *fmixr;  // [L][E]
    const double *decay, *bonus;                       // [L][E]
    const double *expdecay;                            // [L][E] exp(decay), tabulated at load
    const float *emb;                                  // [V][E]
    const double *ones;                                // [E] of 1.0 (batched prefill: "no token shift")
    double *sxy, *sdd;                                 // [slots][L][E] token-shift state (replicated)
    double *x;                                         // [E] residual stream after the last layer (tests)
    Ctrl *ctrl;
    const unsigned long long *stream;                  // device-resident token stream (feed_mode 2)
    Diag *diag;                                        // mapped host memory
    // The exchange block of this rank (one allocation, peer-mapped by the other ranks). Offsets are the
    // same on every rank: xch[g] + off is rank g's copy as seen from here (xch[rank] = the local one).
    unsigned char *xch[kMaxRanks];
    unsigned int off_stat[2];   // [kRep][2][grid] tagged doubles: slice sums, slice Q (LN1 / LN_out, LN2)
    unsigned int off_off[5];    // [kRep][3][grid] tagged doubles: partial offset sums per vector (kvr, out, rk, v, head)
    unsigned int off_max[5];    // [kRep][3][grid] tagged f32: slice max |xs| per vector
    unsigned int off_vec[5];    // f32+tag vectors (kvr 3E, out Er, rk 2E, v 4Er, head E)
    unsigned int off_in[2];     // [G][E] tagged doubles: partial sums from every rank (out-proj, ffn-V)
    unsigned int off_sr;        // [E] tagged f32: sigmoid(ffn r) of every channel
    unsigned int off_arg;       // [G][grid] tagged {logit, index}
    unsigned int off_done;      // [G][grid] tagged completion flags
    unsigned int off_logits;    // [V] f32
    unsigned long long off_saa, off_sbb; // [slots][L][E] f64 WKV state (every rank holds all channels)
    unsigned long long *trace;  // optional [grid][kTraceMax] globaltimer stamps (debug), or nullptr
    unsigned long long *ptrace; // optional [2][grid][kTileTraceMax]: tile issue / tile ready times (debug)
    // ---- generate launches only (k_token<.., GEN = true>; greedy = 1: arg-max, 0: typical sampler) ----
    // (kept behind every other field: the offsets the other instantiations read do not move)
    unsigned int off_smp;       // [kRep][3][grid] tagged doubles: per-CTA sampler partials (max, sum exp, sum exp^e)
    int exponent;               // uint8(1 / temp) of the reference sampler: 0 = uniform draw
    int n_stop;                 // stop ids in `stop`
    double margin_min;          // a sampled token whose uniform lies closer than this to a boundary halts the run
    const double *uniforms;     // [n] the uniforms of the run, indexed by ctrl->pos
    unsigned long long *gen_tokens; // [n] token of step ctrl->pos
    double *gen_margins;        // [n] its margin (typical)
    unsigned long long stop[kMaxStop];
};

// ---------------------------------------------------------------------------------------
// PTX helpers
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ unsigned long long globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok)
                 : "r"(bar), "r"(parity)
                 : "memory");
    return ok != 0;
}
// ---- thread-block cluster helpers (distributed shared memory) ---------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// shared-window address `addr` of this CTA -> the same location in CTA `rank` of the cluster (shared::cluster window)
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
// 4-byte store into another CTA's shared memory that reports its bytes to an mbarrier of THAT CTA: whoever waits
// for the barrier's phase sees the data - no fence on either side (a release at cluster scope costs microseconds
// here: it drains everything the thread has in flight)
__device__ __forceinline__ void st_async32(uint32_t remote_addr, uint32_t v, uint32_t remote_bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(remote_addr), "r"(v), "r"(remote_bar) : "memory");
}
// arrive on an mbarrier of another CTA of the cluster, no ordering implied
__device__ __forceinline__ void mbar_arrive_remote(uint32_t remote_bar) {
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote_bar) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() { // every thread of every CTA of the cluster
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// non-blocking test of an mbarrier phase
__device__ __forceinline__ bool mbar_test_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok)
                 : "r"(bar), "r"(parity)
                 : "memory");
    return ok != 0;
}
// 1-D bulk TMA: global -> shared, completion signalled as transaction bytes on `bar`.
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
                 "[%0], [%1], %2, [%3], %4;" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
// weights (signed bytes) x activation digits (unsigned / signed bytes)
__device__ __forceinline__ int dp4a_su(uint32_t a, uint32_t b, int c) {
    int d;
    asm("dp4a.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ int dp4a_ss(uint32_t a, uint32_t b, int c) {
    int d;
    asm("dp4a.s32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
// Asynchronous 8- / 4-byte copies global -> shared (LDGSTS): epilogue parameters are parked in shared
// memory while the GEMV core has the registers.
__device__ __forceinline__ void cp_async8(void *smem, const void *gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async4(void *smem, const void *gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_all;" ::: "memory"); }
// Identity the optimiser cannot see through (keeps loop-invariant addresses from being rematerialised
// or strength-reduced into dozens of live 64-bit induction pointers inside the GEMV core).
__device__ __forceinline__ int opaque(int v) {
    asm volatile("" : "+r"(v));
    return v;
}
__device__ __forceinline__ uint32_t opaque(uint32_t v) {
    asm volatile("" : "+r"(v));
    return v;
}
__device__ __forceinline__ size_t opaque(size_t v) {
    asm volatile("" : "+l"(v));
    return v;
}

// clock read that the compiler keeps between the computation of `a`, `b` and everything that uses them afterwards
__device__ __forceinline__ long long clock_after(double &a, double &b) {
    long long t;
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(t), "+d"(a), "+d"(b));
    return t;
}
__device__ __forceinline__ void tok_sync() { // named barrier 1: the eight consumer warps
    asm volatile("bar.sync 1, %0;" ::"n"(kConsumers) : "memory");
}
__device__ __forceinline__ void own_sync() { // named barrier 2: warps 0 and 1 (the slice owners)
    asm volatile("bar.sync 2, 64;" ::: "memory");
}

// Fixed-shape (deterministic) warp reductions; every lane receives the result.
// __syncwarp() first: after a divergent branch (if (lane == 0) ..., a trace stamp) the lanes of a warp run
// independently until something reconverges them; ptxas guards every shuffle sequence with BRA.DIV and a
// diverged warp takes a WARPSYNC.COLLECTIVE path that costs ~250 cycles PER SHUFFLE (measured: 2.5 us for
// two interleaved f64 trees instead of 0.1 us).
__device__ __forceinline__ double warp_sum(double v) {
    __syncwarp();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Quantiser scale (decode kernel and batched path alike): 1 / m * kQMax without the IEEE division, whose range
// check sends most calls into a ~100-instruction slow path here (ncu source view: 3 divisions = 870 cycles per
// gather). Hardware reciprocal + one Newton step, then one multiplication - the same bits in every thread of every
// CTA, and that is all the quantiser needs (the dequantisation scale m / kQMax is computed separately, in double).
__device__ __forceinline__ float quant_scale(float m) {
    if (!(m > 0.0f)) return 0.0f;
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(m));
    r = fmaf(r, fmaf(-m, r, 1.0f), r);
    float inv = (float)kQMax * r;
    // |q| <= kQMax needs m * inv < kQMax + 0.5 exactly (the fma is exact to one rounding of a small number)
    for (int k = 0; k < 3; ++k)
        if (fmaf(m, inv, -(float)kQMax) >= 0.5f) inv = __uint_as_float(__float_as_uint(inv) - 1u);
    return inv;
}

// ---------------------------------------------------------------------------------------
// Shared-memory carve-up (dynamic shared memory, 128-byte aligned base)
// ---------------------------------------------------------------------------------------
struct Smem {
    uint8_t *ring;       // stages * tile_bytes
    uint8_t *planes;     // limb planes
    long long *res64;    // [kMaxRowsPerCta] exact integer row totals
    double *scal;        // [16]: [0..2] S of vector v, [3..5] offset sum of vector v, [6..7] mean / std,
                         //       [8] trace counters, [10..15] scratch
    uint32_t *wmax;      // [kWarps][4] per-warp maxima of the gather
    uint64_t *full;      // [stages]
    uint64_t *empty;     // [stages]
    double *xown;        // [kMaxSlice] this CTA's slice of the residual stream
    float *srown;        // [kMaxSlice] sigmoid(ffn r) of the slice (G == 1)
    double *pd;          // [kMaxSlice][8] epilogue parameters of the slice owners, staged with cp.async
    float *pf;           // [kMaxSlice][8]
    float *pk;           // [kMaxKeys][2]  ffn-V scale / offset of the own key channels
    long long *clk;      // [16] debug cycle counters (set_option dbg=4)
    uint64_t *cbar;      // [2] cluster mbarriers: [0] every CTA of the cluster has read its limb planes, [1] the planes are written
    uint32_t *gmax;      // [4] max |xs| of the vectors of the current gather (atomicMax of the warps' parts), [3] boundary flag
    double *osum;        // [kWarps][3] the warps' parts of the offset sums
};

__host__ __device__ inline size_t smem_fixed_bytes() {
    return kMaxRowsPerCta * 8 + 16 * 8 + kWarps * 4 * 4 + 2 * kMaxStages * 8 + kMaxSlice * (8 + 4 + 64 + 32) + kMaxKeys * 8 + 128 + 128 + 16 + 16 + kWarps * 3 * 8;
}
__host__ __device__ inline size_t smem_bytes(int stages, int tile_bytes, int plane_cap) {
    return (size_t)stages * tile_bytes + plane_cap + smem_fixed_bytes();
}

__device__ __forceinline__ Smem carve(uint8_t *base, const Params &p) {
    Smem s;
    s.ring = base;
    uint8_t *q = base + (size_t)p.stages * p.tile_bytes;
    s.planes = q;
    q += p.plane_cap;
    s.res64 = reinterpret_cast<long long *>(q);
    q += kMaxRowsPerCta * sizeof(long long);
    s.scal = reinterpret_cast<double *>(q);
    q += 16 * sizeof(double);
    s.full = reinterpret_cast<uint64_t *>(q);
    q += kMaxStages * sizeof(uint64_t);
    s.empty = reinterpret_cast<uint64_t *>(q);
    q += kMaxStages * sizeof(uint64_t);
    s.xown = reinterpret_cast<double *>(q);
    q += kMaxSlice * sizeof(double);
    s.pd = reinterpret_cast<double *>(q);
    q += kMaxSlice * 8 * sizeof(double);
    s.pf = reinterpret_cast<float *>(q);
    q += kMaxSlice * 8 * sizeof(float);
    s.pk = reinterpret_cast<float *>(q);
    q += kMaxKeys * 2 * sizeof(float);
    s.srown = reinterpret_cast<float *>(q);
    q += kMaxSlice * sizeof(float);
    s.wmax = reinterpret_cast<uint32_t *>(q);
    q += kWarps * 4 * sizeof(uint32_t);
    s.clk = reinterpret_cast<long long *>(q);
    q += 16 * sizeof(long long);
    s.cbar = reinterpret_cast<uint64_t *>(q);
    q += 2 * sizeof(uint64_t);
    s.gmax = reinterpret_cast<uint32_t *>(q);
    q += 4 * sizeof(uint32_t);
    s.osum = reinterpret_cast<double *>(q);
    return s;
}

} // namespace rk
