// token_kernel.cuh — the persistent one-token kernel: one CTA per SM, the whole forward of one token
// in ONE launch, on one GPU or on G GPUs that decode the same stream together.
//
// Reference mapping: cuda_rwkv_parralel (include/rwkv/cuda/rwkv.cu:493-593) = embedding + LN0 (513-524),
// per layer LN1 + mixatt (535-540), K/V/R GEMVs (542), WKV (544-545), out-proj + residual (548-553),
// LN2 + mixffn (557-562), ffn R/K GEMVs + sigmoid / relu^2 (566-573), ffn V + residual (574-577), then
// LN_out + head (585-589).
//
// Structure
//   * Each CTA owns a fixed slice of the residual stream (kept in shared memory for the whole token) and
//     does the elementwise work (layernorm, token shift, WKV, residual adds) for that slice only.
//   * A producer lane streams this CTA's weight rows HBM -> shared memory through a ring of bulk-TMA tiles.
//     Weights do not depend on activations, so it never waits for anything but a free ring stage and
//     keeps HBM busy while the consumer warps exchange vectors.
//   * Eight consumer warps: warp w takes unit w (one row segment) of every tile, activation limbs in
//     registers, 12 IDP.4A per 128-bit LDS, REDUX for the exact int32 totals.
//   * CTAs exchange small vectors as self-tagged words through L2 (exchange.cuh): no grid barrier, no
//     atomics, a reader proceeds as soon as the words it needs carry the current epoch.
//
// Dataflow of one layer (-> = tagged exchange inside one GPU, => = partial sums across GPUs, G > 1 only):
//   slice stats -> [LN1, token shift, own slice] -> xk,xv,xr -> [K,V,R rows of own channels; WKV] -> rwkv
//   -> [out-proj rows of own slice] => [residual; slice stats] -> [LN2, token shift] -> xr,xk
//   -> [ffn-R rows of own channels, ffn-K rows; sigmoid, relu^2] -> k4 -> [ffn-V rows of own slice] =>
//   [residual] ...   then slice stats -> [LN_out] -> xh -> [head rows] -> logits (+ arg-max).
#pragma once
#include "exchange.cuh"

namespace rk {

#ifndef RK_CORE_INLINE
#define RK_CORE_INLINE __forceinline__
#endif

// Position in the shared-memory ring: stage index + parity of the current pass over the ring.
struct RingPos {
    uint32_t stage, phase;
    __device__ __forceinline__ void advance(uint32_t stages) {
        if (++stage == stages) {
            stage = 0;
            phase ^= 1;
        }
    }
};

// Slice ownership of CTA b of nb (per rank). Residual elements are global indices and the same on every
// rank; channels, key channels and vocabulary rows are relative to the rank's shard.
struct Slices {
    int e0, ne; // residual-stream elements = rows of out-proj / ffn-V
    int c0, nc; // att channels of this rank = rows of K, V, R, ffn-R
    int k0, nk; // ffn key channels of this rank = rows of ffn-K
    int v0, nv; // vocabulary rows of this rank
};
__host__ __device__ inline void split_rows(int M, int b, int nb, int &r0, int &n) {
    // M * nb < 2^32 for every matrix here (M <= 50277, nb <= 160): 32-bit unsigned division
    r0 = (int)(((unsigned int)M * (unsigned int)b) / (unsigned int)nb);
    n = (int)(((unsigned int)M * (unsigned int)(b + 1)) / (unsigned int)nb) - r0;
}
__host__ __device__ inline Slices make_slices(int E, int Er, int Vr, int b, int nb) {
    Slices s;
    split_rows(E, b, nb, s.e0, s.ne);
    split_rows(Er, b, nb, s.c0, s.nc);
    split_rows(4 * Er, b, nb, s.k0, s.nk);
    split_rows(Vr, b, nb, s.v0, s.nv);
    return s;
}

// ---- producer ----------------------------------------------------------------------------------------
// Weights are row-major [out][in] int8. A tile is exactly eight work units; a unit is one row segment
// (rows of <= E bytes: one unit per row, eight rows per tile; ffn-V rows of 4*Er bytes: four units per
// row, two rows per tile), so consumer warp w always takes unit w of every tile.
//
// The schedule of one CTA is a fixed sequence of tiles: per layer the subs K, V, R (own channels), out-proj
// (own slice), ffn-R (own channels), ffn-K (own key channels), ffn-V (own slice), then the head rows. Two
// cursors walk it: `cp` issues the bulk copies into the ring (bounded by free stages and by `window` copies in
// flight), `pf` runs `pf_dist` tiles further ahead and only asks L2 to fetch the bytes
// (cp.async.bulk.prefetch.L2). The shared-memory ring holds at most 3.7 us of HBM time; a phase boundary
// takes longer than that, so without the second cursor HBM idles in every boundary and the following phase
// starts from an empty pipe. With it HBM streams continuously into L2 (126 MB) and the ring refills from
// L2 at the consumers' pace.
struct TileCursor {
    int l, s;           // layer (== L_run: head), sub inside the layer
    int r, nr, tr;      // next row inside the sub, rows of the sub, rows per tile
    int N;              // bytes per row
    const int8_t *base; // first row of the sub
};
struct TileRef {
    const int8_t *ptr;
    uint32_t bytes;
};
// (inlined: the producer warp runs with 40 registers after setmaxnreg; a separately compiled function does not know that)
// Sub `s` of layer `l` -> cursor fields (base pointer of the own rows, bytes per row, rows per tile, row count).
__device__ __forceinline__ void load_sub(const Params &p, const Slices &sl, TileCursor &c) {
    const int E = p.E, Er = p.Er;
    c.r = 0;
    if (c.l >= p.L_run) {
        c.N = E; c.tr = 8; c.nr = c.l == p.L_run ? sl.nv : 0;
        c.base = p.whead + (size_t)sl.v0 * E;
        return;
    }
    const size_t mc = (size_t)c.l * Er * E; // one column-split matrix [Er][E]
    switch (c.s) {
    case 0: c.N = E; c.tr = 8; c.nr = sl.nc; c.base = p.wk + mc + (size_t)sl.c0 * E; break;
    case 1: c.N = E; c.tr = 8; c.nr = sl.nc; c.base = p.wv + mc + (size_t)sl.c0 * E; break;
    case 2: c.N = E; c.tr = 8; c.nr = sl.nc; c.base = p.wr + mc + (size_t)sl.c0 * E; break;
    case 3: c.N = Er; c.tr = 8; c.nr = sl.ne; c.base = p.wo + mc + (size_t)sl.e0 * Er; break;
    case 4: c.N = E; c.tr = 8; c.nr = sl.nk; c.base = p.wfk + 4 * mc + (size_t)sl.k0 * E; break; // ffn K before ffn R
    case 5: c.N = E; c.tr = 8; c.nr = sl.nc; c.base = p.wfr + mc + (size_t)sl.c0 * E; break;
    default: c.N = 4 * Er; c.tr = 8 / p.vseg; c.nr = sl.ne; c.base = p.wfv + 4 * mc + (size_t)sl.e0 * 4 * Er; break;
    }
}
// The tile under the cursor, then advance. Returns false at the end of the token's schedule.
__device__ __forceinline__ bool next_tile(const Params &p, const Slices &sl, TileCursor &c, TileRef &t) {
    while (c.r >= c.nr) { // next sub
        if (c.l >= p.L_run) {
            if (c.l > p.L_run) return false;
            ++c.l; // past the head: the end
            c.nr = 0;
            return false;
        }
        if (++c.s == 7) {
            c.s = 0;
            ++c.l;
        }
        load_sub(p, sl, c);
    }
    t.ptr = c.base + (size_t)c.r * c.N;
    t.bytes = (uint32_t)(min(c.tr, c.nr - c.r) * c.N);
    c.r += c.tr;
    return true;
}

// `window`: at most that many bulk copies of this CTA are in flight (issued, not landed). The memory
// system serves the SMs' copies in order, so everything in flight queues AHEAD of the small latency-
// critical loads of an exchange: 5 x 32 KB per SM is 3.7 us of queue at the HBM rate.
template <bool TRACE>
__device__ __forceinline__ void produce_token(const Params &p, const Smem &sm, const Slices &sl) {
    unsigned long long *const ptrace = TRACE ? p.ptrace : nullptr;
    // evict_first keeps the weight stream from displacing the exchange words and the per-layer
    // parameters in L2 (measured in round 1: evict_normal costs 15 %).
    const uint64_t pol = policy_evict_first();
    const uint32_t ring = smem_u32(sm.ring), full0 = smem_u32(sm.full), empty0 = smem_u32(sm.empty);
    RingPos rp{0, 0}, wp{0, 0};
    TileCursor cp, pf;
    cp.l = 0;
    cp.s = 0;
    load_sub(p, sl, cp);
    pf = cp;
    bool pf_live = true;
    int tcount = 0, landed = 0, ahead = 0; // tiles issued; tiles known to have landed; lead of the prefetch cursor over the copy cursor
    const volatile uint32_t *const quiet_flag = reinterpret_cast<volatile uint32_t *>(sm.gmax + 3);
    TileRef t;
    // The pending tile of the copy cursor. A non-blocking loop: top up the L2 prefetches, retire landed copies,
    // issue the pending copy when a ring stage is free and the in-flight window allows it.
    Waiter wt = waiter_begin();
    for (;;) {
        // While the consumers wait for exchanged words (`quiet`), everything this SM has in flight queues ahead of
        // their loads (0.75 us per 32 KB tile) and every prefetch competes with them in L2: keep at most `bwindow`
        // copies in flight and prefetch nothing. Epilogues, quantisation and the GEMV itself are not latency-bound:
        // there the window is `window` copies and L2 is kept `pf_dist` tiles ahead, so HBM keeps streaming.
        while (pf_live && ahead < 1) { // the prefetch cursor never falls behind the copy cursor
            TileRef q;
            pf_live = next_tile(p, sl, pf, q);
            if (!pf_live) break;
            if (p.pf_dist > 0 && ahead >= 1) // (the tile the copy cursor takes next is fetched by the copy itself)
                // default L2 policy: with evict_first the stream of newer prefetches would evict the oldest ones - the
                // tiles about to be consumed; the consuming copy then marks the lines evict_first
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(q.ptr), "r"(q.bytes) : "memory");
            ++ahead;
        }
        if (!next_tile(p, sl, cp, t)) break;
        --ahead;
        for (;;) { // until the pending tile is issued
            while (landed < tcount && mbar_test_wait(full0 + 8 * wp.stage, wp.phase)) {
                wp.advance((uint32_t)p.stages);
                ++landed;
            }
            const int win = *quiet_flag != 0u ? p.bwindow : p.window;
            // first pass over the ring: a fresh mbarrier reports the "previous" phase as complete
            const bool slot_free = mbar_test_wait(empty0 + 8 * rp.stage, rp.phase ^ 1);
            if (tcount - landed < win && slot_free) break;
            // The ring is full (the consumers are in a boundary) and nobody waits for exchanged words: HBM would idle.
            // Only then ask L2 for tiles further ahead - while the ring still takes copies, a prefetch of a far tile
            // would only delay the near ones (same queue, same HBM).
            if (!slot_free && *quiet_flag == 0u && pf_live && ahead < p.pf_dist + 1) {
                TileRef q;
                pf_live = next_tile(p, sl, pf, q);
                if (pf_live) {
                    if (p.pf_dist > 0) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(q.ptr), "r"(q.bytes) : "memory");
                    ++ahead;
                }
            } else {
                __nanosleep(40);
            }
            if (waiter_tick(p, wt)) wait_expired(p, kDiagRingEmpty, 0, 0, (unsigned int)tcount, (unsigned int)landed, 0ull);
        }
        const uint32_t fb = full0 + 8 * rp.stage;
        mbar_expect_tx(fb, t.bytes);
        bulk_g2s(ring + rp.stage * (uint32_t)p.tile_bytes, t.ptr, t.bytes, fb, pol);
        if (ptrace != nullptr && tcount < kTileTraceMax) ptrace[(size_t)blockIdx.x * kTileTraceMax + tcount] = globaltimer();
        ++tcount;
        rp.advance((uint32_t)p.stages);
    }
}

// ---- consumer core -----------------------------------------------------------------------------------
// Exact int32 dot products of one 16-byte chunk against the three limb planes (two chains per plane).
__device__ __forceinline__ void dot_chunk(const uint4 w, const uint4 a0, const uint4 a1, const uint4 a2, int (&acc)[6]) {
    acc[0] = dp4a_su(w.x, a0.x, acc[0]);
    acc[2] = dp4a_su(w.x, a1.x, acc[2]);
    acc[4] = dp4a_ss(w.x, a2.x, acc[4]);
    acc[1] = dp4a_su(w.y, a0.y, acc[1]);
    acc[3] = dp4a_su(w.y, a1.y, acc[3]);
    acc[5] = dp4a_ss(w.y, a2.y, acc[5]);
    acc[0] = dp4a_su(w.z, a0.z, acc[0]);
    acc[2] = dp4a_su(w.z, a1.z, acc[2]);
    acc[4] = dp4a_ss(w.z, a2.z, acc[4]);
    acc[1] = dp4a_su(w.w, a0.w, acc[1]);
    acc[3] = dp4a_su(w.w, a1.w, acc[3]);
    acc[5] = dp4a_ss(w.w, a2.w, acc[5]);
}

// Consumer side of one streamed sub-matrix: warp w takes unit w of every tile. All arguments are plain
// values in registers (the hot loop takes them through opaque()).
// N: bytes per row; nseg: segments per row (1, 2 or 4; a tile is 8 / nseg rows); planes: shared address of limb plane 0 of this sub's
// activation vector (planes 1, 2 at +N, +2N); res: shared address of this sub's int64 [row][nseg] totals.
// CPL: 16-byte chunks per lane that hold the limbs of one segment (N / nseg <= CPL * 512).
// BOUNDED = false: the segment is exactly CPL * 512 bytes - straight-line code, no predicates.
// BOUNDED = true : any shorter segment (narrow models, the Er-byte rows of a tensor-parallel rank): the
//                  chunk loop ends at the first chunk index past the segment (a warp-uniform branch).
template <int CPL, bool BOUNDED>
__device__ __forceinline__ RingPos consume_sub(const Params &p, uint32_t ring, uint32_t full0, uint32_t empty0, uint32_t tile_bytes,
                                               uint32_t stages, uint32_t planes, uint32_t res, int N, int nseg, int nr, RingPos rp,
                                               int warp, int lane, unsigned long long *ptrace, int *tile_cnt) {
    const int sh = nseg >> 1;    // log2(nseg) for nseg = 1, 2, 4
    const int tr = 8 >> sh;      // rows per tile
    const int seg_len = N >> sh;
    const int nchunks = seg_len >> 4;
    // this warp's unit inside every tile: (row warp / nseg, segment warp % nseg)
    const int seg = warp & (nseg - 1), rl = warp >> sh;
    const uint32_t unit_off = (uint32_t)(rl * N + seg * seg_len + lane * 16);
    const int ntiles = (nr + tr - 1) / tr;
    if (ntiles <= 0) return rp;
    uint4 a0[CPL], a1[CPL], a2[CPL];
    {
        const uint32_t pl = planes + (uint32_t)(seg * seg_len);
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
            const int c = lane + 32 * i;
            if (!BOUNDED || c < nchunks) {
                a0[i] = lds128(pl + c * 16);
                a1[i] = lds128(pl + N + c * 16);
                a2[i] = lds128(pl + 2 * N + c * 16);
            } else {
                a0[i] = a1[i] = a2[i] = make_uint4(0, 0, 0, 0);
            }
        }
    }
    uint32_t dst = res + (uint32_t)((rl * nseg + seg) * 8);
    int row = rl;
    // The three warp sums of a row are issued after its IDPs and stored one tile later, behind the next row's IDPs:
    // in the plain order (sum, move out of the uniform register, combine, store) a tenth of the loop's samples were
    // waits for the REDUX results.
    int s0 = 0, s1 = 0, s2 = 0;
    uint32_t sdst = 0;
    bool spend = false;
    for (int t = 0; t < ntiles; ++t) {
        mbar_wait(p, full0 + 8 * rp.stage, rp.phase, kDiagRingFull);
        if (ptrace != nullptr && threadIdx.x == 0) {
            const int c = *tile_cnt;
            if (c < kTileTraceMax) ptrace[((size_t)gridDim.x + blockIdx.x) * kTileTraceMax + c] = globaltimer();
            *tile_cnt = c + 1;
        }
        const bool act = row < nr;
        int acc[6] = {0, 0, 0, 0, 0, 0};
        if (act) {
            const uint32_t wrow = ring + rp.stage * tile_bytes + unit_off;
            if (!BOUNDED) {
                uint4 w[CPL];
#pragma unroll
                for (int i = 0; i < CPL; ++i) w[i] = lds128(wrow + i * 512);
#pragma unroll
                for (int i = 0; i < CPL; ++i) dot_chunk(w[i], a0[i], a1[i], a2[i], acc);
            } else {
                // chunks of this lane: lane + 32 i < nchunks; whole groups of 32 chunks are warp-uniform
#pragma unroll
                for (int i = 0; i < CPL; ++i) {
                    if (32 * i < nchunks) {
                        const uint4 w = lane + 32 * i < nchunks ? lds128(wrow + i * 512) : make_uint4(0, 0, 0, 0);
                        dot_chunk(w, a0[i], a1[i], a2[i], acc);
                    }
                }
            }
        }
        if (spend && lane == 0) {
            const long long tot = (((long long)s2 << 8) + (long long)s1) * 256 + (long long)s0;
            asm volatile("st.shared.u64 [%0], %1;" ::"r"(sdst), "l"(tot) : "memory");
        }
        spend = act;
        sdst = dst;
        if (act) {
            s0 = __reduce_add_sync(0xffffffffu, acc[0] + acc[1]);
            s1 = __reduce_add_sync(0xffffffffu, acc[2] + acc[3]);
            s2 = __reduce_add_sync(0xffffffffu, acc[4] + acc[5]);
        }
        dst += 8 * 8;
        row += tr;
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8 * rp.stage);
        rp.advance(stages);
    }
    if (spend && lane == 0) {
        const long long tot = (((long long)s2 << 8) + (long long)s1) * 256 + (long long)s0;
        asm volatile("st.shared.u64 [%0], %1;" ::"r"(sdst), "l"(tot) : "memory");
    }
    return rp;
}

// ---- activation quantiser -----------------------------------------------------------------------------
// q = round(xs * inv) as a 23-bit two's complement integer (|q| <= 2^22 - 1); the three limb planes are
// its three low BYTES: bytes 0 and 1 are unsigned digits, byte 2 is the signed top digit. Rounding goes
// through the float adder (1.5 * 2^23 + x has ulp 1: the low mantissa bits are the integer) - no F2I;
// four elements are transposed into the planes with seven PRMTs.
__device__ __forceinline__ uint32_t round_q(float xs, float inv) {
    return __float_as_uint(fmaf(xs, inv, 12582912.0f)) - 0x4B400000u;
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
// four elements -> their word in each of the three limb planes
struct PlaneWords {
    uint32_t w0, w1, w2;
};
__device__ __forceinline__ PlaneWords quantize4(const uint4 f, float inv) {
    const uint32_t t0 = round_q(untag_f32(f.x), inv), t1 = round_q(untag_f32(f.y), inv);
    const uint32_t t2 = round_q(untag_f32(f.z), inv), t3 = round_q(untag_f32(f.w), inv);
    const uint32_t lo01 = __byte_perm(t0, t1, 0x5140), lo23 = __byte_perm(t2, t3, 0x5140);
    const uint32_t hi01 = __byte_perm(t0, t1, 0x0062), hi23 = __byte_perm(t2, t3, 0x0062);
    return PlaneWords{__byte_perm(lo01, lo23, 0x5410), __byte_perm(lo01, lo23, 0x7632), __byte_perm(hi01, hi23, 0x5410)};
}

// ---- debug tracing --------------------------------------------------------------------------------------
// Executed by the whole of warp 0 with predicated stores: a branch taken by lane 0 alone would split the warp,
// and a split warp pays ~100 cycles for every later shuffle (the first version of this function made the
// reductions that followed a stamp look 10x slower than they are).
__device__ __forceinline__ void trace_stamp(unsigned long long *trace, double *scal, int ctid) {
    if (trace != nullptr && ctid < 32) {
        const uint32_t cnt = smem_u32(scal + 8);
        int c;
        asm volatile("ld.shared.s32 %0, [%1];" : "=r"(c) : "r"(cnt) : "memory");
        const unsigned long long t = globaltimer();
        unsigned long long *dst = trace + (size_t)blockIdx.x * kTraceMax + (c < kTraceMax ? c : kTraceMax - 1);
        __syncwarp(); // every lane has read the counter
        asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.s32 p, %0, 0;\n\t@p st.global.u64 [%1], %2;\n\t@p st.shared.s32 [%3], %4;\n\t}"
                     ::"r"(ctid), "l"(dst), "l"(t), "r"(cnt), "r"(c < kTraceMax ? c + 1 : c)
                     : "memory");
    }
}

// ---- gather: exchanged vectors -> limb planes --------------------------------------------------------
// The `nvec` vectors of length N (contiguous f32+tag words at `vec`) were written by their slice owners.
// Every thread polls the first 16 bytes of its share until they carry this epoch, then fetches the rest
// in one batch (one L2 round trip when everything has arrived, which is the normal case: the owners
// publish within a fraction of a microsecond of each other), re-reads whatever was not there yet, takes
// the per-vector max |xs| over the block and quantises from registers into the limb planes
// (vector v -> planes + v*3*N). Warp 7 also sums the owners' partial offset sums (OffRec) in a fixed
// order. Result: scal[v] = S_v (value of one integer step), scal[3+v] = sum_j x_j * oc_j.
// Every CTA starts at a different offset so that the CTAs do not hit the same L2 lines together.
// Inlined ONCE (the phase loop of the kernel has a single call site): as a separate function it would be
// compiled against the 168-register launch budget instead of the consumers' 232 and spill.
constexpr int kGatherMax = 20; // 16-byte groups per thread: 256 x 20 x 4 >= 4 * 5120
__device__ __forceinline__ void gather(const Params &p, const Smem &sm, const float *vec, const TaggedDouble *offrec,
                                       const unsigned long long *maxrec, int nvec,
                                       int N, uint32_t tag, unsigned int layer, int ctid, int gk, unsigned long long *trace) {
    const uint32_t tag2 = tag & 3u;
    const int ng = N >> 2;        // groups per vector
    const int total = nvec * ng;  // <= 256 * kGatherMax
    // The C CTAs of a thread-block cluster split the gather: CTA r of the cluster fetches and quantises the r-th
    // part of the concatenated vectors and writes the limb-plane words into the shared memory of all C CTAs
    // (st.shared::cluster). All 148 SMs pulling the same 16..64 KB out of L2 is what bounds the exchange (L2
    // bandwidth, tools/latbench.cu part 3) and the quantisation is ~2 us of ALU work per phase: both shrink by C.
    // (Starting every CTA at a different offset of the vector was measured slower than walking it in the same order.)
    const int C = p.cluster;
    const int part = total / C;   // N is a multiple of 16: total is a multiple of 4
    const int base = (C > 1 ? (int)cluster_ctarank() * part : 0) + ctid;
    const int cnt = (part - ctid + kConsumers - 1) / kConsumers; // groups of this thread (may be <= 0)
    const uint4 *src = reinterpret_cast<const uint4 *>(vec);
    auto index = [&](int i) { return base + kConsumers * i; };
    const uint4 absent = make_uint4(tag2, tag2, tag2, tag2); // +0.0f carrying the tag: a slot this thread does not have
    uint4 f[kGatherMax];
    Waiter wt = waiter_begin();
    f[0] = absent;
    // poll_first 2: meet at the block barrier first - the owners of THIS CTA have published by then, and the
    // CTAs run in step, so one batch of loads normally finds everything (one L2 round trip, no polling
    // traffic while the owners still compute); 1: poll the first 16 bytes, then the batch; 0: batch at once.
    if (ctid == 0) *reinterpret_cast<volatile uint32_t *>(sm.gmax + 3) = 1u; // latency-bound window: the producer goes quiet
    if (p.poll_first == 2) tok_sync();
    trace_stamp(trace, sm.scal, ctid); // G1: block met
    if (cnt > 0 && p.poll_first != 1) f[0] = ld_vec4(src + index(0));
    if (cnt > 0 && p.poll_first == 1) {
        const uint4 *s0 = src + index(0);
        f[0] = ld_vec4(s0);
        while (!vec4_ok(f[0], tag2)) {
            if (waiter_tick(p, wt)) wait_expired(p, kDiagVec, layer, (unsigned int)nvec, tag2, f[0].x & 3u, (unsigned long long)index(0));
            f[0] = ld_vec4(s0);
        }
    }
    __syncwarp();
#pragma unroll
    for (int i = 1; i < kGatherMax; ++i) {
        f[i] = absent;
        if (i < cnt) f[i] = ld_vec4(src + index(i));
    }
    // The owners' records (partial offset sums, slice maxima), spread over the eight warps: warp w takes records
    // w, w+8, ... (one per lane). Only the maxima are needed before the quantisation: one REDUX per vector and an
    // atomicMax in shared memory; the f64 sums are reduced after the quantisation, off the critical path.
    const int lane = ctid & 31, wq = ctid >> 5;
    const int rec = wq + kWarps * lane;
    const bool has_rec = rec < (int)gridDim.x;
    const unsigned long long none = tag64(0u, tag);
    const TaggedDouble *const orec = offrec + (size_t)(blockIdx.x % kRep) * 3 * gridDim.x + rec; // this CTA's replica
    const unsigned long long *const mrec = maxrec + (size_t)(blockIdx.x % kRep) * 3 * gridDim.x + rec;
    unsigned long long ra[3], rb[3], rm[3];
#pragma unroll
    for (int v = 0; v < 3; ++v) {
        ra[v] = rb[v] = rm[v] = none;
        if (has_rec && v < nvec) {
            ld_pair(orec + v * (int)gridDim.x, ra[v], rb[v], false);
            rm[v] = ld_word(mrec + v * (int)gridDim.x, false);
        }
    }
    for (;;) {
        bool bad = false;
#pragma unroll
        for (int v = 0; v < 3; ++v) {
            if (!tags_ok(ra[v], rb[v], tag)) {
                ld_pair(orec + v * (int)gridDim.x, ra[v], rb[v], false);
                bad = true;
            }
            if ((uint32_t)(rm[v] >> 32) != tag) {
                rm[v] = ld_word(mrec + v * (int)gridDim.x, false);
                bad = true;
            }
        }
        if (!__any_sync(0xffffffffu, bad)) break; // warp-uniform exit (see slice_stats)
        if (waiter_tick(p, wt)) wait_expired(p, kDiagOff, layer, (unsigned int)nvec, tag, (unsigned int)(ra[0] >> 32), (unsigned long long)rec);
    }
#pragma unroll
    for (int v = 0; v < 3; ++v) {
        const uint32_t mm = __reduce_max_sync(0xffffffffu, (uint32_t)rm[v]);
        if (lane == 0 && v < nvec) atomicMax(sm.gmax + v, mm);
    }
    // late words: re-read until every group carries the tag
    for (;;) {
        bool bad = false;
#pragma unroll
        for (int i = 0; i < kGatherMax; ++i) {
            if (!vec4_ok(f[i], tag2)) {
                f[i] = ld_vec4(src + index(i));
                bad = true;
            }
        }
        if (!__any_sync(0xffffffffu, bad)) break; // warp-uniform exit (see slice_stats)
        if (waiter_tick(p, wt)) wait_expired(p, kDiagVec, layer, (unsigned int)nvec, tag2, 99u, (unsigned long long)base);
    }
    trace_stamp(trace, sm.scal, ctid); // all words here
    trace_stamp(trace, sm.scal, ctid); // G3
    tok_sync(); // the maxima of all warps are in shared memory
    trace_stamp(trace, sm.scal, ctid); // G4
    const bool probe = (p.dbg & 8) != 0; // cycle counters of the steps below, thread 0, summed over the token
    long long pc[6];
    auto tick = [&](int k) {
        if (probe) asm volatile("mov.u64 %0, %%clock64;" : "=l"(pc[k])::"memory");
    };
    tick(0);
    if (ctid == 0) *reinterpret_cast<volatile uint32_t *>(sm.gmax + 3) = 0u; // the exchange loads are back: the producer may open its window
    float inv0, inv1, inv2;
    {   // scale of vector v (the same bits in every thread and every CTA)
        const float m0 = __uint_as_float(sm.gmax[0]), m1 = __uint_as_float(sm.gmax[1]), m2 = __uint_as_float(sm.gmax[2]);
        inv0 = quant_scale(m0);
        inv1 = quant_scale(m1);
        inv2 = quant_scale(m2);
        if (ctid < 3) sm.scal[ctid] = (double)(ctid == 0 ? m0 : ctid == 1 ? m1 : m2) * (1.0 / (double)kQMax);
    }
    const uint32_t pl0 = smem_u32(sm.planes);
    tick(1);
    if (C == 1) {
#pragma unroll
        for (int i = 0; i < kGatherMax; ++i) {
            if (i < cnt) {
                // element 4*gg of the concatenated vectors sits 4*gg + v*2N bytes into the planes (3N bytes per vector)
                const int gg = index(i);
                const int v = (gg >= ng) + (gg >= 2 * ng);
                const float iv = v == 0 ? inv0 : v == 1 ? inv1 : inv2;
                const PlaneWords w = quantize4(f[i], iv);
                const uint32_t a = pl0 + (uint32_t)(4 * gg + 2 * v * N);
                sts32(a, w.w0);
                sts32(a + (uint32_t)N, w.w1);
                sts32(a + 2u * (uint32_t)N, w.w2);
            }
        }
    } else {
        // every CTA of the cluster has finished the GEMV that read its planes (signalled after that GEMV)
        if (gk > 0) mbar_wait(p, smem_u32(sm.cbar), (uint32_t)(gk - 1) & 1u, kDiagPlanesFree);
        const uint32_t me = cluster_ctarank(), bar1 = smem_u32(sm.cbar + 1);
        uint32_t plr[4], barr[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            plr[r] = mapa(pl0, (uint32_t)(r < C ? r : 0));
            barr[r] = mapa(bar1, (uint32_t)(r < C ? r : 0));
        }
#pragma unroll
        for (int i = 0; i < kGatherMax; ++i) {
            if (i < cnt) {
                const int gg = index(i);
                const int v = (gg >= ng) + (gg >= 2 * ng);
                const float iv = v == 0 ? inv0 : v == 1 ? inv1 : inv2;
                const PlaneWords w = quantize4(f[i], iv);
                const uint32_t o = (uint32_t)(4 * gg + 2 * v * N);
                sts32(pl0 + o, w.w0);
                sts32(pl0 + o + (uint32_t)N, w.w1);
                sts32(pl0 + o + 2u * (uint32_t)N, w.w2);
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    if (r < C && r != (int)me) {
                        st_async32(plr[r] + o, w.w0, barr[r]);
                        st_async32(plr[r] + o + (uint32_t)N, w.w1, barr[r]);
                        st_async32(plr[r] + o + 2u * (uint32_t)N, w.w2, barr[r]);
                    }
                }
            }
        }
    }
    tick(2);
    {   // this warp's part of the offset sums (fixed trees), then warps 0..7 in order by thread v
        double t0 = has_rec ? pair_to_double(ra[0], rb[0]) : 0.0, t1 = has_rec ? pair_to_double(ra[1], rb[1]) : 0.0,
               t2 = has_rec ? pair_to_double(ra[2], rb[2]) : 0.0;
        __syncwarp();
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            t0 += __shfl_xor_sync(0xffffffffu, t0, o);
            t1 += __shfl_xor_sync(0xffffffffu, t1, o);
            t2 += __shfl_xor_sync(0xffffffffu, t2, o);
        }
        if (lane == 0) {
            sm.osum[wq * 3 + 0] = t0;
            sm.osum[wq * 3 + 1] = t1;
            sm.osum[wq * 3 + 2] = t2;
        }
    }
    tick(3);
    if (C == 1) {
        tok_sync();
    } else {
        // "planes written": this CTA's eight warps arrive after their own stores; the other CTAs' words arrive as
        // transaction bytes (12 per group of four elements) of their st.async
        __syncwarp();
        const uint32_t bar1 = smem_u32(sm.cbar + 1);
        if (lane == 0) {
            if (wq == 0) mbar_expect_tx(bar1, 12u * (uint32_t)(total - part));
            else mbar_arrive(bar1);
        }
        mbar_wait(p, bar1, (uint32_t)gk & 1u, kDiagPlanesReady);
    }
    tick(4);
    if (ctid < 3) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) t += sm.osum[w * 3 + ctid];
        sm.scal[3 + ctid] = t;  // read by the epilogue, after the GEMV and its barrier
        sm.gmax[ctid] = 0u;     // for the next gather
    }
    tick(5);
    if (probe && ctid == 0) {
        for (int k = 0; k < 5; ++k) sm.clk[8 + k] += pc[k + 1] - pc[k];
        sm.clk[13] += 1;
    }
    trace_stamp(trace, sm.scal, ctid); // planes ready
}

// ---- slice statistics -----------------------------------------------------------------------------------
// Layernorm statistics of the whole residual stream from per-CTA {S = sum x, Q = sum (x - c0)^2} in double,
// where c0 is a reference point every CTA already knows: the mean of the previous statistics (0 at the
// start of a token). The residual moves the mean only a little, so Q carries no cancellation, and
//   sum_j (x_j - c)^2 = Q - 2 (c - c0)(S - E c0) + E (c - c0)^2
// for the reference's f32-rounded mean c is exactly its second pass (rwkv.cu:432-450); the two accumulators
// are rounded to f32 like its float atomics (412-465, 43-44). Called by warps 0 and 1 (the slice owners);
// xown holds the slice. The reader's work after the records arrive is two shuffle reductions and a dozen
// scalar operations - this sits on the critical path of every layer twice.
// Returns mean and 1 / sqrt(var) (unbiased, no epsilon); c0 is updated to the new mean.
struct StatsOut {
    double mean, rstd;
};
static __device__ __noinline__ StatsOut slice_stats(const Params &p, const double *xown, double *scal, long long *clkp, volatile uint32_t *quiet,
                                             TaggedDouble *recs, int ne, uint32_t tag, unsigned int layer, int ctid, double c0,
                                             unsigned long long *trace) {
    struct {
        const double *xown;
        double *scal;
        long long *clk;
    } sm{xown, scal, clkp};
    own_sync(); // xown complete
    if (ctid == 0) *quiet = 1u; // latency-bound window: the producer goes quiet (token_kernel.cuh: produce_token)
    trace_stamp(trace, sm.scal, ctid); // S1: owners synchronised
    if (ctid < 32) {
        const int lane = ctid;
        const int nb = (int)gridDim.x;
        // Every CTA reads every record: 148 x 32 lanes on the same few L2 lines serialise there (measured 1.6 us
        // for one batch of loads). The writer stores kRep copies, reader b takes copy b % kRep.
        TaggedDouble *const sums = recs + (size_t)(blockIdx.x % kRep) * 2 * nb, *const qs = sums + nb; // [nb] each
        const double v0 = lane < ne ? sm.xown[lane] : 0.0, v1 = lane + 32 < ne ? sm.xown[lane + 32] : 0.0;
        const double d0 = lane < ne ? v0 - c0 : 0.0, d1 = lane + 32 < ne ? v1 - c0 : 0.0;
        double s = v0 + v1, q = d0 * d0 + d1 * d1;
        __syncwarp(); // reconverge (see warp_sum in common.cuh)
        const bool clk = (p.dbg & 4) != 0;
        long long tc0 = 0, tc1 = 0, tc2 = 0, tc3 = 0, tc4 = 0;
        if (clk) tc0 = clock_after(s, q);
        if ((p.dbg & 2) && trace != nullptr) { // debug: split the segment
            if (__double_as_longlong(q) == 0x7ff8000000000001ll) s = 0.0; // (consume q before the stamp)
            trace_stamp(trace, sm.scal, ctid);
            __syncwarp();
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { // two independent trees, interleaved
            s += __shfl_xor_sync(0xffffffffu, s, o);
            q += __shfl_xor_sync(0xffffffffu, q, o);
        }
        if ((p.dbg & 2) && trace != nullptr) {
            if (__double_as_longlong(q) == 0x7ff8000000000001ll) s = 0.0;
            trace_stamp(trace, sm.scal, ctid);
        }
        if (clk) tc1 = clock_after(s, q);
        __syncwarp();
        if (lane < kRep) {
            st_tagged_double(&recs[(size_t)lane * 2 * nb + blockIdx.x], s, tag, false);
            st_tagged_double(&recs[(size_t)lane * 2 * nb + nb + blockIdx.x], q, tag, false);
        }
        trace_stamp(trace, sm.scal, ctid); // S2: own record published
        // every CTA's record: all in flight at once (r = lane, lane+32, ...), re-read what has not arrived
        constexpr int kPer = (kMaxGrid + 31) / 32;
        const unsigned long long none = tag64(0u, tag);
        unsigned long long a[kPer], b[kPer], c[kPer], d[kPer];
#pragma unroll
        for (int i = 0; i < kPer; ++i) {
            a[i] = b[i] = c[i] = d[i] = none;
            if (lane + 32 * i < nb) {
                ld_pair(&sums[lane + 32 * i], a[i], b[i], false);
                ld_pair(&qs[lane + 32 * i], c[i], d[i], false);
            }
        }
        Waiter w = waiter_begin();
        trace_stamp(trace, sm.scal, ctid); // S3: loads issued
        for (;;) {
            bool bad = false;
#pragma unroll
            for (int i = 0; i < kPer; ++i) {
                if (!tags_ok(a[i], b[i], tag)) {
                    ld_pair(&sums[lane + 32 * i], a[i], b[i], false);
                    bad = true;
                }
                if (!tags_ok(c[i], d[i], tag)) {
                    ld_pair(&qs[lane + 32 * i], c[i], d[i], false);
                    bad = true;
                }
            }
            // warp-uniform exit: lanes that leave a loop at different iterations stay split, and a split warp
            // pays ~100 cycles for every shuffle afterwards, __syncwarp() or not (measured: 1850 vs 260 cycles)
            if (!__any_sync(0xffffffffu, bad)) break;
            if (waiter_tick(p, w)) wait_expired(p, kDiagStats, layer, 0, tag, (unsigned int)(a[0] >> 32), (unsigned long long)lane);
        }
        if (ctid == 0) *quiet = 0u;
        trace_stamp(trace, sm.scal, ctid); // S4: every record here
        double st = 0.0, qt = 0.0;
#pragma unroll
        for (int i = 0; i < kPer; ++i) { // ascending record index per lane, then fixed trees: deterministic
            st += pair_to_double(a[i], b[i]);
            qt += pair_to_double(c[i], d[i]);
        }
        if (clk) tc2 = clock_after(st, qt);
        __syncwarp();
        if (clk) tc3 = clock_after(st, qt);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            st += __shfl_xor_sync(0xffffffffu, st, o);
            qt += __shfl_xor_sync(0xffffffffu, qt, o);
        }
        if (clk) {
            tc4 = clock_after(st, qt);
            if (lane == 0) {
                long long *ck = sm.clk + ((layer & 0x8000u) ? 8 : 0); // the debug "cold" call counts separately
                ck[0] += tc1 - tc0; // first pair of trees
                ck[1] += tc2 - tc1; // publish + records
                ck[2] += tc3 - tc2; // __syncwarp
                ck[3] += tc4 - tc3; // second pair of trees
                ck[4] += 1;
            }
        }
        if (lane == 0) {
            const double Ed = (double)p.E;
            const float mean_acc = (float)st;
            const double mean_f = (double)(mean_acc / (float)p.E); // the variance kernel's float / float mean
            const double dc = mean_f - c0;
            double m2 = qt - 2.0 * dc * (st - Ed * c0) + Ed * dc * dc;
            if (m2 < 0.0) m2 = 0.0;
            const float sd = sqrtf((float)m2 / (float)(p.E - 1));
            sm.scal[6] = (double)mean_acc / Ed;
            sm.scal[7] = 1.0 / (double)sd;
        }
        trace_stamp(trace, sm.scal, ctid); // S5: statistics computed
    }
    own_sync();
    return StatsOut{sm.scal[6], sm.scal[7]};
}

// Partial offset sums and the largest |xs| of this CTA's slice (data in the first `nact` consumer threads, NV
// values each) -> its records. Fixed reduction shape: shuffle tree per warp, then warps 0..nw-1 in order.
// Called by every consumer warp; warps without data return at once. (NV > 1 only for slice owners: <= 2 warps.)
// mx: bit patterns of non-negative floats (they order like unsigned integers).
template <int NV>
__device__ __forceinline__ void publish_slice(const Smem &sm, TaggedDouble *recs, unsigned long long *mrecs, double (&of)[NV],
                                              uint32_t (&mx)[NV], uint32_t tag, int ctid, int nact) {
    const int nw = nact > 0 ? (nact + 31) >> 5 : 1; // an empty slice still publishes zeros
    const int w = ctid >> 5;
    if (w >= nw) return;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        of[k] = warp_sum(of[k]);
        mx[k] = __reduce_max_sync(0xffffffffu, mx[k]);
    }
    double *scr = sm.scal + 10; // [nw - 1][NV] <= 6 doubles
    uint32_t *mscr = sm.wmax;   // [kWarps][4]
    if (nw > 1) {
        if ((ctid & 31) == 0 && w > 0) {
#pragma unroll
            for (int k = 0; k < NV; ++k) {
                scr[(w - 1) * NV + k] = of[k];
                mscr[w * 4 + k] = mx[k];
            }
        }
        asm volatile("bar.sync 3, %0;" ::"r"(nw * 32) : "memory");
        if (w == 0) { // every lane of warp 0 adds the other warps' parts in the same order
            for (int i = 1; i < nw; ++i) {
#pragma unroll
                for (int k = 0; k < NV; ++k) {
                    of[k] += scr[(i - 1) * NV + k];
                    mx[k] = max(mx[k], mscr[i * 4 + k]);
                }
            }
        }
    }
    if (w == 0 && (ctid & 31) < kRep) { // lane r stores replica r: [kRep][3][grid]
#pragma unroll
        for (int k = 0; k < NV; ++k) {
            const size_t at = ((size_t)(ctid & 31) * 3 + k) * gridDim.x + blockIdx.x;
            st_tagged_double(&recs[at], of[k], tag, false);
            st_word(&mrecs[at], tag64(mx[k], tag), false);
        }
    }
}

// Sum over the G ranks of the partial result `part` of residual element j (a row-split GEMV): store it into
// every peer's inbox, wait for the peers' parts, add in rank order (identical on every rank). Called by whole
// warps (`valid` = this lane owns an element); the polling loop is warp-uniform.
static __device__ __noinline__ double peer_sum(const Params &p, unsigned int off_in, int j, double part, bool valid, uint32_t tag,
                                        unsigned int layer) {
    if (valid)
        for (int g = 0; g < p.G; ++g)
            if (g != p.rank) st_tagged_double(xch_at<TaggedDouble>(p, g, off_in) + ((size_t)p.rank * p.E + j), part, tag, true);
    const TaggedDouble *in = xch_at<TaggedDouble>(p, p.rank, off_in);
    const unsigned long long none = tag64(0u, tag);
    unsigned long long a[kMaxRanks], b[kMaxRanks];
#pragma unroll
    for (int g = 0; g < kMaxRanks; ++g) { // all peers' words in flight at once
        a[g] = b[g] = none;
        if (valid && g < p.G && g != p.rank) ld_pair(&in[(size_t)g * p.E + j], a[g], b[g], true);
    }
    Waiter w = waiter_begin();
    for (;;) {
        bool bad = false;
#pragma unroll
        for (int g = 0; g < kMaxRanks; ++g) {
            if (!tags_ok(a[g], b[g], tag)) {
                ld_pair(&in[(size_t)g * p.E + j], a[g], b[g], true);
                bad = true;
            }
        }
        if (!__any_sync(0xffffffffu, bad)) break;
        if (waiter_tick(p, w)) wait_expired(p, kDiagPeerSum, layer, 0, tag, (unsigned int)(a[p.rank == 0 ? 1 : 0] >> 32), (unsigned long long)j);
    }
    double tot = 0.0;
#pragma unroll
    for (int g = 0; g < kMaxRanks; ++g) // rank order, the own part in its place: identical on every rank
        if (g < p.G) tot += g == p.rank ? part : pair_to_double(a[g], b[g]);
    return tot;
}

// sigmoid(ffn r) of residual element j, published by the owner of that channel (any rank). Whole warps.
static __device__ __noinline__ float peer_sr(const Params &p, int j, bool valid, uint32_t tag, unsigned int layer) {
    const unsigned long long *srp = xch_at<unsigned long long>(p, p.rank, p.off_sr) + j;
    unsigned long long a = tag64(0u, tag);
    Waiter w = waiter_begin();
    for (;;) {
        bool bad = false;
        if (valid) {
            a = ld_word(srp, true);
            bad = (uint32_t)(a >> 32) != tag;
        }
        if (!__any_sync(0xffffffffu, bad)) break;
        if (waiter_tick(p, w)) wait_expired(p, kDiagSr, layer, 0, tag, (unsigned int)(a >> 32), (unsigned long long)j);
    }
    return __uint_as_float((uint32_t)a);
}

// ---- the typical sampler over the head's logits (generate launches) ------------------------------------
// The token is the one typical_with_u(logits, temp, u) returns (include/rwkv/sampler/typical.h): p_i ~ (exp(l_i) /
// sum)^e with e = uint8(1 / temp), the first index whose sequential cumulative probability reaches u, cp_last
// forced to 1. For e >= 1 the normalised distribution is softmax(e * l), so no CTA needs the global sum of exp(l)
// before it can sum its powers: CTA b publishes {m_b = max of its logits, A_b = sum exp(l - m_b), B_b = sum exp(e
// (l - m_b))} in ONE exchange (a second exchange for the global sum would add another all-to-all round trip to
// every token) and every reader rescales to the global maximum M, so nothing overflows whatever e is. Every CTA
// builds the prefix P over the CTAs from the same words with the same fixed-shape scan, so all agree on every
// boundary and exactly one finds u in its interval (P_b, P_b+1] (CTA 0's closed at 0, the last one open to the
// top: cp_last = 1 and u < 1). That CTA scans its own rows (block scan of the logits recomputed from the integer row
// totals in shared memory) and finishes the step: token and margin into the run's arrays at ctrl->pos, the token
// into ctrl->next, and the halt flag when the margin is below margin_min or the token is a stop id. The device sums
// differ from the host's sequential ones by ~1e-13, hence the margin; where the host's own arithmetic leaves the
// range of doubles (its sum of exp(l) over the vocabulary overflows once max l > 709.78 - ln(V); (exp(l) / sum)^e
// underflows for a large e: A_b gives the host's sum), and where rounding left u above the claiming CTA's own
// running sum, the margin is reported as -1: the step always halts and the host decides with its own arithmetic.
__device__ __forceinline__ bool is_stop(const Params &p, unsigned long long t) {
    bool stop = false;
#pragma unroll
    for (int k = 0; k < kMaxStop; ++k) stop = stop || (k < p.n_stop && p.stop[k] == t);
    return stop;
}
__device__ __forceinline__ void sample_head(const Params &p, const Smem &sm, int v0, int nv, int ctid) {
    // the step index: written by this step's finishing CTA only after it has this CTA's record (published below)
    const unsigned long long pos = p.ctrl->pos;
    const int lane = ctid & 31, w = ctid >> 5, nb = (int)gridDim.x, b = (int)blockIdx.x;
    const int e = p.exponent;
    const double de = (double)e;
    auto logit = [&](int i) { return (float)(sm.scal[0] * (double)sm.res64[i] + sm.scal[3]); };
    auto power = [&](double d) { return e == 0 ? 1.0 : e == 1 ? exp(d) : exp(de * d); }; // exp(l - m)^e
    double *sh = sm.osum;                                        // [kWarps * 3] scratch
    uint32_t *wm = sm.wmax;                                      // [kWarps]
    float mx = -INFINITY;
    for (int i = ctid; i < nv; i += kConsumers) mx = fmaxf(mx, logit(i));
    __syncwarp();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) sh[w] = (double)mx;
    tok_sync();
    double m = sh[0];
    for (int k = 1; k < kWarps; ++k) m = fmax(m, sh[k]);
    if (!(m > -INFINITY)) m = 0.0; // no finite logit: the sums below are NaN or 0 and the host decides
    tok_sync();
    double a = 0.0, bs = 0.0;
    for (int i = ctid; i < nv; i += kConsumers) {
        const double d = (double)logit(i) - m;
        a += exp(d);
        bs += power(d);
    }
    a = warp_sum(a);
    bs = warp_sum(bs);
    if (lane == 0) {
        sh[w * 3 + 0] = a;
        sh[w * 3 + 1] = bs;
    }
    tok_sync();
    if (w == 0) {
        double A = 0.0, B = 0.0;
        for (int k = 0; k < kWarps; ++k) { // warps in order: the same bits in every lane
            A += sh[k * 3 + 0];
            B += sh[k * 3 + 1];
        }
        TaggedDouble *const recs = xch_at<TaggedDouble>(p, p.rank, p.off_smp);
        if (lane < kRep) {
            st_tagged_double(&recs[((size_t)lane * 3 + 0) * nb + b], m, p.tk, false);
            st_tagged_double(&recs[((size_t)lane * 3 + 1) * nb + b], A, p.tk, false);
            st_tagged_double(&recs[((size_t)lane * 3 + 2) * nb + b], B, p.tk, false);
        }
        // lane l holds records l*kPer .. l*kPer + kPer - 1 (contiguous: the prefix is a lane-local sum + one warp scan)
        constexpr int kPer = (kMaxGrid + 31) / 32;
        const TaggedDouble *const rd = recs + (size_t)(b % kRep) * 3 * nb;
        const unsigned long long none = tag64(0u, p.tk);
        unsigned long long ra[kPer][3], rb[kPer][3];
#pragma unroll
        for (int i = 0; i < kPer; ++i) {
            const int r = lane * kPer + i;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                ra[i][k] = rb[i][k] = none;
                if (r < nb) ld_pair(&rd[(size_t)k * nb + r], ra[i][k], rb[i][k], false);
            }
        }
        Waiter wt = waiter_begin();
        for (;;) {
            bool bad = false;
#pragma unroll
            for (int i = 0; i < kPer; ++i)
#pragma unroll
                for (int k = 0; k < 3; ++k)
                    if (!tags_ok(ra[i][k], rb[i][k], p.tk)) {
                        ld_pair(&rd[(size_t)k * nb + lane * kPer + i], ra[i][k], rb[i][k], false);
                        bad = true;
                    }
            if (!__any_sync(0xffffffffu, bad)) break; // warp-uniform exit (see slice_stats)
            if (waiter_tick(p, wt)) wait_expired(p, kDiagSample, (unsigned int)p.L_run, 0, p.tk, (unsigned int)(ra[0][0] >> 32), (unsigned long long)lane);
        }
        double M = -INFINITY;
#pragma unroll
        for (int i = 0; i < kPer; ++i)
            if (lane * kPer + i < nb) M = fmax(M, pair_to_double(ra[i][0], rb[i][0]));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) M = fmax(M, __shfl_xor_sync(0xffffffffu, M, o));
        double P[kPer], run = 0.0, asum = 0.0;
#pragma unroll
        for (int i = 0; i < kPer; ++i) {
            double wgt = 0.0;
            if (lane * kPer + i < nb) {
                const double mb = pair_to_double(ra[i][0], rb[i][0]);
                const double Bb = pair_to_double(ra[i][2], rb[i][2]);
                wgt = e == 0 ? Bb : exp(de * (mb - M)) * Bb;
                asum += exp(mb - M) * pair_to_double(ra[i][1], rb[i][1]);
            }
            P[i] = run;
            run += wgt;
        }
        double incl = run;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += y;
        }
        double excl = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane == 0) excl = 0.0;
        const double S = __shfl_sync(0xffffffffu, incl, 31);
        asum = warp_sum(asum);
        double lo = 0.0, hi = 0.0;
#pragma unroll
        for (int i = 0; i < kPer; ++i) {
            const double Pr = excl + P[i]; // the same formula for every record in every CTA
            if (lane * kPer + i == b) lo = Pr;
            if (lane * kPer + i == b + 1) hi = Pr;
        }
        lo = __shfl_sync(0xffffffffu, lo, b / kPer) / S;
        hi = b + 1 < nb ? __shfl_sync(0xffffffffu, hi, (b + 1) / kPer) / S : 2.0;
        const double u = p.uniforms[pos];
        const bool claim = (b == 0 || lo < u) && !(hi < u);
        bool ok = S > 0.0 && S < INFINITY;
        // host: sum of exp(l) <= V exp(M) must stay finite (709.78 = ln of the largest double), exp(l) normal
        if (e >= 1) ok = ok && M <= 709.0 - log((double)kVocab) && M >= -600.0;
        if (e >= 2) ok = ok && log(S) - de * log(asum) > -650.0;
        if (lane == 0) {
            sh[0] = claim ? 1.0 : 0.0;
            sh[1] = lo;
            sh[2] = (e == 0 ? 1.0 : exp(de * (m - M))) / S; // own rows: p_i = exp(l_i - m)^e * f
            sh[3] = u;
            sh[4] = ok ? 1.0 : 0.0;
        }
    }
    tok_sync();
    if (sh[0] == 0.0) return; // block-uniform
    const double f = sh[2], u = sh[3];
    const bool ok = sh[4] != 0.0;
    double carry = sh[1];
    tok_sync(); // sh is reused below
    int found = -1;
    double fmargin = 0.0;
    for (int c0 = 0; c0 < nv; c0 += kConsumers) {
        const int i = c0 + ctid;
        const bool valid = i < nv;
        const double pi = valid ? power((double)logit(i) - m) * f : 0.0;
        double x = pi;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        double xex = __shfl_up_sync(0xffffffffu, x, 1);
        if (lane == 0) xex = 0.0;
        if (lane == 31) sh[w] = x;
        tok_sync();
        double woff = 0.0, tot = 0.0;
        for (int k = 0; k < kWarps; ++k) {
            if (k < w) woff += sh[k];
            tot += sh[k];
        }
        const double c = carry + (woff + x), prev = carry + (woff + xex);
        const bool last = b == nb - 1 && i == nv - 1;
        const uint32_t cand = valid && (last || !(c < u)) ? (uint32_t)i : 0xffffffffu;
        const uint32_t wmin = __reduce_min_sync(0xffffffffu, cand);
        if (lane == 0) wm[w] = wmin;
        tok_sync();
        uint32_t first = wm[0];
        for (int k = 1; k < kWarps; ++k) first = min(first, wm[k]);
        if (first != 0xffffffffu) {
            found = (int)first;
            if ((uint32_t)i == first) fmargin = last ? u - prev : fmin(u - prev, c - u);
            break; // block-uniform
        }
        carry = carry + tot;
        tok_sync();
    }
    // rounding left u above this CTA's own running sum (found < 0): no trusted token, the host decides
    const bool writer = found >= 0 ? ctid == found - (found / kConsumers) * kConsumers : ctid == 0;
    if (writer) {
        const unsigned long long t = (unsigned long long)(p.vbase + v0 + (found >= 0 ? found : nv - 1));
        const double margin = !ok || found < 0 ? -1.0 : fmargin;
        p.gen_tokens[pos] = t;
        p.gen_margins[pos] = margin;
        p.ctrl->next = t;
        p.ctrl->pos = pos + 1;
        if (is_stop(p, t) || !(margin >= p.margin_min)) p.ctrl->halt = 1;
    }
}

// CPL: 16-byte chunks per lane of an E-byte row segment (the values instantiated: RK_CPLS); FULL: E == CPL * 512;
// TRACE: with the %globaltimer stamps of tools/trace_token.py (set_option("trace", 1)).
// GEN: a step of rwkv_b200_generate - halted launches exit at entry, the head finishes with the arg-max (p.greedy)
// or the typical sampler and records the step (a separate instantiation: the other launches keep their code).
#define RK_CPLS(X) X(2) X(4) X(6) X(8) X(10)
template <int CPL, bool FULL, bool TRACE, bool GEN = false>
__global__ void __launch_bounds__(kThreads, 1) k_token(const __grid_constant__ Params p) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const Smem sm = carve(smem_raw, p);
    // generate: the halt flag was written by the previous launch; every thread reads it before the barrier below, so
    // the CTA that finishes this step (after every CTA has published) cannot race it
    bool halted = false;
    if constexpr (GEN) halted = p.ctrl->halt != 0;
    if (threadIdx.x == 0) {
        for (int i = 0; i < p.stages; ++i) {
            mbar_init(smem_u32(&sm.full[i]), 1);
            mbar_init(smem_u32(&sm.empty[i]), kWarps);
        }
        mbar_init(smem_u32(&sm.cbar[0]), (uint32_t)p.cluster);          // one arrival per CTA of the cluster
        mbar_init(smem_u32(&sm.cbar[1]), (uint32_t)kWarps);    // the own consumer warps (+ the peers' st.async bytes)
        mbar_fence_init();
    }
    __syncthreads();
    if constexpr (GEN) {
        if (halted) return; // uniform over the grid: no exchange, no state write, epochs untouched
    }
    if (p.cluster > 1) cluster_sync_all(); // the peers' barriers exist before anybody arrives on them
    const int E = p.E, Er = p.Er;
    const int nb = (int)gridDim.x;
    const Slices sl = make_slices(E, Er, p.Vr, (int)blockIdx.x, nb);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp >= kWarps) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kProducerRegs));
        if (warp == kWarps && lane == 0) produce_token<TRACE>(p, sm, sl);
        return;
    }
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kConsumerRegs));
    const int ctid = threadIdx.x;
    const int ne = sl.ne, nc = sl.nc, nk = sl.nk;
    const bool owner_warps = warp < 2;  // warps 0 and 1 hold the slice owners (ne, nc <= 64)
    const bool mine = ctid < ne;        // this thread owns residual element e0 + ctid
    const bool minec = ctid < nc;       // this thread owns att channel rank*Er + c0 + ctid
    const bool minek = ctid < nk;       // this thread owns ffn key channel rank*4Er + k0 + ctid
    const bool multi = p.G > 1;
    if (ctid == 0) {
        *reinterpret_cast<int *>(sm.scal + 8) = 0;
        *reinterpret_cast<int *>(sm.scal + 9) = 0;
        for (int i = 0; i < 16; ++i) sm.clk[i] = 0;
        for (int i = 0; i < 4; ++i) sm.gmax[i] = 0u;
    }
    unsigned long long *const c_trace = (TRACE && !(p.dbg & 4)) ? p.trace : nullptr;
    auto stamp = [&]() {
        if (TRACE) trace_stamp(c_trace, sm.scal, ctid);
    };
    const int j = sl.e0 + (mine ? ctid : 0);    // residual element (clamped to an owned one)
    const int cl = sl.c0 + (minec ? ctid : 0);  // channel inside the rank's shard (clamped)
    const int cg = p.rank * Er + cl;            // global channel
    const Ctrl *ctrl = p.ctrl;
    unsigned long long token = ctrl->token;
    if (p.feed_mode == 1) token = ctrl->next;
    else if (p.feed_mode == 2) token = p.stream[ctrl->pos];
    const size_t so = (size_t)ctrl->slot * p.L * E; // state slot offset
    unsigned char *const xl = p.xch[p.rank];
    TaggedDouble *const stat0 = reinterpret_cast<TaggedDouble *>(xl + p.off_stat[0]);
    TaggedDouble *const stat1 = reinterpret_cast<TaggedDouble *>(xl + p.off_stat[1]);
    const double *const saa = reinterpret_cast<const double *>(xl + p.off_saa);
    const double *const sbb = reinterpret_cast<const double *>(xl + p.off_sbb);
    double *const pd = sm.pd + (ctid & (kMaxSlice - 1)) * 8; // this owner thread's parameter slots
    float *const pf = sm.pf + (ctid & (kMaxSlice - 1)) * 8;
    float *const pk = sm.pk + (ctid < kMaxKeys ? ctid : 0) * 2;

    RingPos rp{0, 0};
    const uint32_t c_ring = opaque(smem_u32(sm.ring)), c_full = opaque(smem_u32(sm.full)), c_empty = opaque(smem_u32(sm.empty));
    const uint32_t c_planes = opaque(smem_u32(sm.planes)), c_res = opaque(smem_u32(sm.res64));
    const uint32_t c_tile = opaque((uint32_t)p.tile_bytes), c_stages = opaque((uint32_t)p.stages);
    const int c_warp = opaque(warp), c_lane = opaque(lane);
    unsigned long long *const c_ptrace = TRACE ? reinterpret_cast<unsigned long long *>(opaque((size_t)p.ptrace)) : nullptr;
    int *const c_tcnt = reinterpret_cast<int *>(sm.scal + 9);
    // exact integer total of row `i` of the sub whose partials start at res64[off] (nseg per row)
    auto row_total = [&](int off, int i, int nseg) {
        long long t = 0;
        for (int sgm = 0; sgm < nseg; ++sgm) t += sm.res64[off + i * nseg + sgm];
        return (double)t;
    };
    stamp();

    // ---- x = LN0(emb[token]) for the own slice (rwkv.cu:513-524): every CTA takes the statistics of the
    // embedding row itself (two passes with the reference's f32 rounding, rwkv.cu:412-465)
    {
        const float *row = p.emb + (size_t)token * E;
        double *ws = reinterpret_cast<double *>(sm.res64); // res64 is free until the first GEMV
        double sacc = 0.0;
        for (int g = ctid; g < (E >> 2); g += kConsumers) {
            const float4 f = *reinterpret_cast<const float4 *>(row + 4 * g);
            sacc += ((double)f.x + (double)f.y) + ((double)f.z + (double)f.w);
        }
        sacc = warp_sum(sacc);
        if (lane == 0) ws[warp] = sacc;
        tok_sync();
        double tot = 0.0;
        for (int w = 0; w < kWarps; ++w) tot += ws[w];
        const float mean_acc = (float)tot;
        const double mean_f = (double)(mean_acc / (float)E);
        double qacc = 0.0;
        for (int g = ctid; g < (E >> 2); g += kConsumers) {
            const float4 f = *reinterpret_cast<const float4 *>(row + 4 * g);
            const double d0 = (double)f.x - mean_f, d1 = (double)f.y - mean_f, d2 = (double)f.z - mean_f, d3 = (double)f.w - mean_f;
            qacc += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
        }
        qacc = warp_sum(qacc);
        if (lane == 0) ws[16 + warp] = qacc;
        tok_sync();
        double qtot = 0.0;
        for (int w = 0; w < kWarps; ++w) qtot += ws[16 + w];
        const double xmean = (double)mean_acc / (double)E;
        const double x2 = (double)sqrtf((float)qtot / (float)(E - 1));
        if (mine) sm.xown[ctid] = p.ln[j] * (((double)row[j] - xmean) / x2) + p.ln[E + j];
        tok_sync(); // the scratch in res64 is reused by the first GEMV
    }

    double c0 = 0.0; // reference point of the slice statistics: the previous mean (same value on every CTA)
    // Parameters of the slice computation that follows a residual update, parked in this thread's shared
    // slots: LN1 + att token shift of layer l (l < L_run), or LN_out + head scale (l == L_run).
    auto fetch_ln1 = [&](int l) {
        if (l < p.L_run) {
            const size_t lo = (size_t)l * E + j;
            cp_async8(pd + 0, p.ln + (size_t)(4 * l + 2) * E + j);
            cp_async8(pd + 1, p.ln + (size_t)(4 * l + 3) * E + j);
            cp_async8(pd + 2, p.mixk + lo);
            cp_async8(pd + 3, p.mixv + lo);
            cp_async8(pd + 4, p.mixr + lo);
            cp_async8(pd + 5, p.sxy + so + lo);
            cp_async4(pf + 0, p.rk + lo);
            cp_async4(pf + 1, p.rv + lo);
            cp_async4(pf + 2, p.rr + lo);
            cp_async4(pf + 3, p.ock + lo);
            cp_async4(pf + 4, p.ocv + lo);
            cp_async4(pf + 5, p.ocr + lo);
        } else {
            cp_async8(pd + 0, p.ln + (size_t)(4 * p.L + 2) * E + j);
            cp_async8(pd + 1, p.ln + (size_t)(4 * p.L + 3) * E + j);
            cp_async4(pf + 0, p.rhead + j);
            cp_async4(pf + 1, p.ochead + j);
        }
    };
    // Slice statistics -> LN1 + token shift of layer l -> publish xk, xv, xr (rwkv.cu:535-540); or, after
    // the last layer, LN_out -> publish the head input (rwkv.cu:585-588). Warps 0 and 1.
    auto slice_to_att = [&](int l) {
        const uint32_t ep = p.ep0 + 1u + (uint32_t)l;
        const StatsOut so1 = slice_stats(p, sm.xown, sm.scal, sm.clk, reinterpret_cast<volatile uint32_t *>(sm.gmax + 3), stat0, ne, ep, (unsigned int)l, ctid, c0, c_trace);
        const double xmean = so1.mean, rstd = so1.rstd;
        c0 = xmean;
        stamp();
        cp_async_wait();
        if (l < p.L_run) {
            float *const vec_kvr = reinterpret_cast<float *>(xl + p.off_vec[0]);
            double of[3] = {0, 0, 0};
            uint32_t mx[3] = {0u, 0u, 0u};
            if (mine) {
                const uint32_t t2 = ep & 3u;
                const double mk = pd[2], mv = pd[3], mr = pd[4], st = pd[5];
                const double ln = pd[0] * ((sm.xown[ctid] - xmean) * rstd) + pd[1];
                const float fk = (float)(mk * ln + (1.0 - mk) * st);
                const float fv = (float)(mv * ln + (1.0 - mv) * st);
                const float fr = (float)(mr * ln + (1.0 - mr) * st);
                const float xk = (float)((double)fk * (double)pf[0]);
                const float xv = (float)((double)fv * (double)pf[1]);
                const float xr = (float)((double)fr * (double)pf[2]);
                const uint32_t bk = tag_f32(xk, t2), bv = tag_f32(xv, t2), br = tag_f32(xr, t2);
                st_f32(vec_kvr + j, bk);
                st_f32(vec_kvr + E + j, bv);
                st_f32(vec_kvr + 2 * E + j, br);
                mx[0] = bk & 0x7ffffffcu; mx[1] = bv & 0x7ffffffcu; mx[2] = br & 0x7ffffffcu;
                of[0] = (double)fk * (double)pf[3];
                of[1] = (double)fv * (double)pf[4];
                of[2] = (double)fr * (double)pf[5];
                p.sxy[so + (size_t)l * E + j] = ln; // only the owner ever reads or writes this element
            }
            publish_slice<3>(sm, reinterpret_cast<TaggedDouble *>(xl + p.off_off[0]), reinterpret_cast<unsigned long long *>(xl + p.off_max[0]), of, mx, ep, ctid, ne);
        } else {
            float *const vec_h = reinterpret_cast<float *>(xl + p.off_vec[4]);
            double of[1] = {0};
            uint32_t mx[1] = {0u};
            if (mine) {
                const float f = (float)(pd[0] * ((sm.xown[ctid] - xmean) * rstd) + pd[1]);
                const float xh = (float)((double)f * (double)pf[0]);
                const uint32_t bh = tag_f32(xh, p.tk & 3u);
                st_f32(vec_h + j, bh);
                mx[0] = bh & 0x7ffffffcu;
                of[0] = (double)f * (double)pf[1];
                p.x[j] = sm.xown[ctid]; // residual stream after the last layer (debug / tests)
            }
            publish_slice<1>(sm, reinterpret_cast<TaggedDouble *>(xl + p.off_off[4]), reinterpret_cast<unsigned long long *>(xl + p.off_max[4]), of, mx, p.tk, ctid, ne);
        }
        stamp();
    };
    if (owner_warps) {
        fetch_ln1(0);
        slice_to_att(0);
    }

    // ---- the phase loop: 5 phases per layer, then the head. One call site each for the gather and the
    // GEMV core keeps the layer body small enough for the instruction cache.
    // Phase 3 (ffn R) gathers nothing: its input was quantised together with ffn K's in phase 2 and its result
    // (the sigmoid gate) is needed only after ffn V, so its 2.4 us of streaming run while the relu^2 keys of
    // phase 2 travel to the other CTAs - phase 4's gather finds them in place.
    const int n_iter = 5 * p.L_run + 1;
    int l = 0, ph = 0, gk = 0; // layer, phase, gathers so far
    for (int it = 0; it < n_iter; ++it) {
        if (opaque(it) == 5 * p.L_run) ph = 5;
        const int xi = ph < 3 ? ph : ph - 1; // index of the phase's exchange areas (kvr, o, rk, k4, head)
        const size_t lo = (size_t)l * E;
        const uint32_t ep = p.ep0 + 1u + (uint32_t)l;
        // -------- what this phase gathers and streams ---------------------------------------------
        int nvec, N, nseg, nsub, nr0, sub0 = 0;
        uint32_t tag;
        switch (ph) {
        case 0: nvec = 3; N = E; nseg = 1; nsub = 3; nr0 = nc; tag = ep; break;               // K, V, R
        case 1: nvec = 1; N = Er; nseg = 1; nsub = 1; nr0 = ne; tag = ep; break;              // out-proj
        case 2: nvec = 2; N = E; nseg = 1; nsub = 1; nr0 = nk; sub0 = 1; tag = ep; break;     // ffn K (input vector 1 of the gather)
        case 3: nvec = 0; N = E; nseg = 1; nsub = 1; nr0 = nc; tag = ep; break;               // ffn R (input vector 0, already quantised)
        case 4: nvec = 1; N = 4 * Er; nseg = p.vseg; nsub = 1; nr0 = ne; tag = ep; break;     // ffn V: rows of 4E/G bytes in segments of <= E
        default: nvec = 1; N = E; nseg = 1; nsub = 1; nr0 = sl.nv; tag = p.tk; break;         // head
        }
        const float *vec = reinterpret_cast<const float *>(xl + p.off_vec[xi]);
        const TaggedDouble *offrec = reinterpret_cast<const TaggedDouble *>(xl + p.off_off[xi]);
        const unsigned long long *maxrec = reinterpret_cast<const unsigned long long *>(xl + p.off_max[xi]);
        // -------- park the epilogue's parameters in shared memory ------------------------------------
        if (ph == 0) {
            if (owner_warps) { // WKV of channel cg (clamped: an idle thread reads a valid address)
                cp_async8(pd + 0, saa + so + lo + cg);
                cp_async8(pd + 1, sbb + so + lo + cg);
                cp_async8(pd + 2, p.decay + lo + cg);
                cp_async8(pd + 3, p.bonus + lo + cg);
                cp_async8(pd + 4, p.expdecay + lo + cg);
                cp_async4(pf + 0, p.ro + lo + cg);
                cp_async4(pf + 1, p.oco + lo + cg);
            }
        } else if (ph == 1) {
            if (owner_warps) { // LN2 + ffn token shift of element j
                cp_async8(pd + 0, p.ln + (size_t)(4 * (l + 1)) * E + j);
                cp_async8(pd + 1, p.ln + (size_t)(4 * (l + 1) + 1) * E + j);
                cp_async8(pd + 2, p.fmixk + lo + j);
                cp_async8(pd + 3, p.fmixr + lo + j);
                cp_async8(pd + 4, p.sdd + so + lo + j);
                cp_async4(pf + 0, p.rfr + lo + j);
                cp_async4(pf + 1, p.rfk + lo + j);
                cp_async4(pf + 2, p.ocfr + lo + j);
                cp_async4(pf + 3, p.ocfk + lo + j);
            }
        } else if (ph == 2) {
            if (minek) { // ffn-V scale / offset of the own key channel
                const size_t ko = (size_t)l * 4 * E + (size_t)p.rank * 4 * Er + sl.k0 + ctid;
                cp_async4(pk + 0, p.rfv + ko);
                cp_async4(pk + 1, p.ocfv + ko);
            }
        } else if (ph == 4) {
            if (owner_warps) fetch_ln1(l + 1);
        }
        // -------- gather + stream ------------------------------------------------------------------
        if (nvec > 0) {
            gather(p, sm, vec, offrec, maxrec, nvec, N, tag, (unsigned int)l, ctid, gk, c_trace);
            ++gk;
        }
        {
            const bool exact = FULL && N == nseg * E; // segment == CPL * 512 bytes
            // results: [sub][row]; ffn K's rows sit behind ffn R's (phase 3 fills those while phase 2's are read)
            uint32_t planes = c_planes + (uint32_t)(sub0 * 3 * N), res = c_res + (uint32_t)(sub0 * nc) * 8u;
            for (int s = 0; s < nsub; ++s) {
                if (exact) rp = consume_sub<CPL, false>(p, c_ring, c_full, c_empty, c_tile, c_stages, planes, res, N, nseg, nr0, rp, c_warp, c_lane, c_ptrace, c_tcnt);
                else rp = consume_sub<CPL, true>(p, c_ring, c_full, c_empty, c_tile, c_stages, planes, res, N, nseg, nr0, rp, c_warp, c_lane, c_ptrace, c_tcnt);
                planes += (uint32_t)(3 * N);
                res += (uint32_t)(nr0 * nseg) * 8u;
            }
        }
        tok_sync();
        // this CTA's limb planes may be overwritten - unless the next phase streams against them without a gather
        // (2 -> 3); nobody gathers after the head
        if (p.cluster > 1 && ctid == 0 && ph != 2 && ph != 5) {
            const uint32_t bar = smem_u32(sm.cbar);
            for (int r = 0; r < p.cluster; ++r) mbar_arrive_remote(mapa(bar, (uint32_t)r));
        }
        stamp();
        cp_async_wait();
        // -------- epilogue ----------------------------------------------------------------------------
        if (ph == 0) {
            // ======== WKV for the own channels (rwkv.cu:544-545) -> rwkv * r_out =========================
            if (owner_warps) {
                double of[1] = {0};
                uint32_t mx[1] = {0u};
                if (minec) {
                    const double aa = pd[0], bb = pd[1], wd = pd[2], ub = pd[3], ew = pd[4]; // exp(decay) is static: tabulated at load
                    const float kf = (float)(sm.scal[0] * row_total(0, ctid, 1) + sm.scal[3]);
                    const float vf = (float)(sm.scal[1] * row_total(nc, ctid, 1) + sm.scal[4]);
                    const float rf = (float)(sm.scal[2] * row_total(2 * nc, ctid, 1) + sm.scal[5]);
                    const double vv = (double)vf;
                    const double e1 = exp(ub + wd + (double)kf);
                    double y = (aa + e1 * vv) / (bb + e1);
                    y = (1.0 / (1.0 + (double)expf(-rf))) * y;
                    const double ek = exp((double)kf);
                    const double naa = (aa + ek * vv) * ew, nbb = (bb + ek) * ew;
                    // every rank keeps the WKV state of all channels (plain peer stores, ordered before the
                    // completion flags at the end of the kernel)
                    for (int g = 0; g < p.G; ++g) {
                        xch_at<double>(p, g, p.off_saa)[so + lo + cg] = naa;
                        xch_at<double>(p, g, p.off_sbb)[so + lo + cg] = nbb;
                    }
                    const float rw = (float)y;
                    const float xo = (float)((double)rw * (double)pf[0]);
                    const uint32_t bo = tag_f32(xo, ep & 3u);
                    st_f32(reinterpret_cast<float *>(xl + p.off_vec[1]) + cl, bo);
                    mx[0] = bo & 0x7ffffffcu;
                    of[0] = (double)rw * (double)pf[1];
                }
                publish_slice<1>(sm, reinterpret_cast<TaggedDouble *>(xl + p.off_off[1]), reinterpret_cast<unsigned long long *>(xl + p.off_max[1]), of, mx, ep, ctid, nc);
            }
        } else if (ph == 1) {
            // ======== residual (rwkv.cu:548-553), then LN2 + token shift (557-562) ========================
            if (owner_warps) {
                double part = mine ? sm.scal[0] * row_total(0, ctid, 1) + sm.scal[3] : 0.0;
                if (multi) part = peer_sum(p, p.off_in[0], j, part, mine, ep, (unsigned int)l);
                if (mine) {
                    const float y = (float)part;
                    const float xf = (float)sm.xown[ctid] + y; // the reference accumulates on an f32 copy of x
                    sm.xown[ctid] = (double)xf;
                }
                stamp();
                const StatsOut so2 = slice_stats(p, sm.xown, sm.scal, sm.clk, reinterpret_cast<volatile uint32_t *>(sm.gmax + 3), stat1, ne, ep, (unsigned int)l, ctid, c0, c_trace);
                const double xmean = so2.mean, rstd = so2.rstd;
                c0 = xmean;
                stamp();
                double of[2] = {0, 0};
                uint32_t mx[2] = {0u, 0u};
                if (mine) {
                    const double fmk = pd[2], fmr = pd[3], fst = pd[4];
                    const double ln = pd[0] * ((sm.xown[ctid] - xmean) * rstd) + pd[1];
                    const float fr = (float)(fmr * ln + (1.0 - fmr) * fst);
                    const float fk = (float)(fmk * ln + (1.0 - fmk) * fst);
                    const float xr = (float)((double)fr * (double)pf[0]);
                    const float xk = (float)((double)fk * (double)pf[1]);
                    float *const vec_rk = reinterpret_cast<float *>(xl + p.off_vec[2]);
                    const uint32_t br = tag_f32(xr, ep & 3u), bk = tag_f32(xk, ep & 3u);
                    st_f32(vec_rk + j, br);
                    st_f32(vec_rk + E + j, bk);
                    mx[0] = br & 0x7ffffffcu; mx[1] = bk & 0x7ffffffcu;
                    of[0] = (double)fr * (double)pf[2];
                    of[1] = (double)fk * (double)pf[3];
                    p.sdd[so + lo + j] = ln;
                }
                publish_slice<2>(sm, reinterpret_cast<TaggedDouble *>(xl + p.off_off[2]), reinterpret_cast<unsigned long long *>(xl + p.off_max[2]), of, mx, ep, ctid, ne);
            }
        } else if (ph == 2) {
            // ======== relu^2 of the own key channels (rwkv.cu:566-573) ====================================
            double of[1] = {0};
            uint32_t mx[1] = {0u};
            if (minek) {
                float a = (float)(sm.scal[1] * row_total(nc, ctid, 1) + sm.scal[4]);
                a = a > 0.0f ? a : 0.0f;
                a = a * a;
                const float xv = (float)((double)a * (double)pk[0]);
                const uint32_t bv = tag_f32(xv, ep & 3u);
                st_f32(reinterpret_cast<float *>(xl + p.off_vec[3]) + sl.k0 + ctid, bv);
                mx[0] = bv & 0x7ffffffcu;
                of[0] = (double)a * (double)pk[1];
            }
            publish_slice<1>(sm, reinterpret_cast<TaggedDouble *>(xl + p.off_off[3]), reinterpret_cast<unsigned long long *>(xl + p.off_max[3]), of, mx, ep, ctid, nk);
        } else if (ph == 3) {
            // ======== sigmoid(ffn r) for the own channels ================================================
            if (minec) {
                const float y = (float)(sm.scal[0] * row_total(0, ctid, 1) + sm.scal[3]);
                const float sr = (float)(1.0 / (1.0 + exp(-(double)y)));
                if (!multi) sm.srown[ctid] = sr; // one GPU: channel owner == residual owner
                else
                    for (int g = 0; g < p.G; ++g) st_word(xch_at<unsigned long long>(p, g, p.off_sr) + cg, tag64(__float_as_uint(sr), ep), true);
            }
        } else if (ph == 4) {
            // ======== residual (rwkv.cu:574-577), then the next layer's LN1 (or LN_out) ====================
            if (owner_warps) {
                double part = mine ? sm.scal[0] * row_total(0, ctid, p.vseg) + sm.scal[3] : 0.0;
                float sr = 0.0f;
                if (multi) {
                    part = peer_sum(p, p.off_in[1], j, part, mine, ep, (unsigned int)l);
                    sr = peer_sr(p, j, mine, ep, (unsigned int)l);
                } else if (mine) {
                    sr = sm.srown[ctid];
                }
                if (mine) {
                    const float kv = (float)part;
                    sm.xown[ctid] = sm.xown[ctid] + (double)(kv * sr);
                }
                stamp();
                slice_to_att(l + 1);
            }
        } else {
            // ======== logits (rwkv.cu:589), arg-max =====================================================
            float best = -INFINITY;
            int bidx = 0x7fffffff;
            for (int i = ctid; i < sl.nv; i += kConsumers) {
                const float y = (float)(sm.scal[0] * row_total(0, i, 1) + sm.scal[3]);
                const int vi = p.vbase + sl.v0 + i;
                for (int g = 0; g < p.G; ++g) xch_at<float>(p, g, p.off_logits)[vi] = y;
                if (y > best) { // i ascending per thread: first maximum kept
                    best = y;
                    bidx = vi;
                }
            }
            if (p.greedy) {
                // block arg-max, first index wins ties
                __syncwarp();
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const float ov2 = __shfl_xor_sync(0xffffffffu, best, o);
                    const int oi = __shfl_xor_sync(0xffffffffu, bidx, o);
                    if (ov2 > best || (ov2 == best && oi < bidx)) {
                        best = ov2;
                        bidx = oi;
                    }
                }
                float *bv = reinterpret_cast<float *>(sm.wmax);
                int *bi = reinterpret_cast<int *>(sm.wmax + 8);
                if (lane == 0) {
                    bv[warp] = best;
                    bi[warp] = bidx;
                }
                tok_sync();
                if (ctid == 0) {
                    for (int w = 1; w < kWarps; ++w)
                        if (bv[w] > best || (bv[w] == best && bi[w] < bidx)) {
                            best = bv[w];
                            bidx = bi[w];
                        }
                    for (int g = 0; g < p.G; ++g)
                        st_pair(xch_at<TaggedDouble>(p, g, p.off_arg) + ((size_t)p.rank * nb + blockIdx.x),
                                tag64(__float_as_uint(best), p.tk), tag64((uint32_t)bidx, p.tk), multi);
                }
                if (blockIdx.x == 0) {
                    // CTA 0 of every rank picks the winner of all G x nb candidates (same result everywhere)
                    const TaggedDouble *cand = xch_at<TaggedDouble>(p, p.rank, p.off_arg);
                    float b2 = -INFINITY;
                    int i2 = 0x7fffffff;
                    Waiter w = waiter_begin();
                    for (int r0 = 0; r0 < p.G * nb; r0 += kConsumers) {
                        const int r = r0 + ctid;
                        unsigned long long a = tag64(0xff800000u, p.tk), b = tag64(0x7fffffffu, p.tk); // (-inf, no index)
                        for (;;) {
                            bool bad = false;
                            if (r < p.G * nb) {
                                ld_pair(&cand[r], a, b, multi);
                                bad = !tags_ok(a, b, p.tk);
                            }
                            if (!__any_sync(0xffffffffu, bad)) break;
                            if (waiter_tick(p, w)) wait_expired(p, kDiagArg, (unsigned int)l, 0, p.tk, (unsigned int)(a >> 32), (unsigned long long)r);
                        }
                        const float v = __uint_as_float((uint32_t)a);
                        const int ix = (int)(uint32_t)b;
                        if (v > b2 || (v == b2 && ix < i2)) {
                            b2 = v;
                            i2 = ix;
                        }
                    }
                    __syncwarp();
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        const float ov2 = __shfl_xor_sync(0xffffffffu, b2, o);
                        const int oi = __shfl_xor_sync(0xffffffffu, i2, o);
                        if (ov2 > b2 || (ov2 == b2 && oi < i2)) {
                            b2 = ov2;
                            i2 = oi;
                        }
                    }
                    tok_sync(); // bv / bi of the first reduction are consumed
                    if (lane == 0) {
                        bv[warp] = b2;
                        bi[warp] = i2;
                    }
                    tok_sync();
                    if (ctid == 0) {
                        for (int w2 = 1; w2 < kWarps; ++w2)
                            if (bv[w2] > b2 || (bv[w2] == b2 && bi[w2] < i2)) {
                                b2 = bv[w2];
                                i2 = bi[w2];
                            }
                        p.ctrl->next = (unsigned long long)(i2 == 0x7fffffff ? 0 : i2);
                        if constexpr (GEN) {
                            const unsigned long long t = (unsigned long long)(i2 == 0x7fffffff ? 0 : i2);
                            const unsigned long long pos = p.ctrl->pos; // this thread is its only writer
                            p.gen_tokens[pos] = t;
                            p.ctrl->pos = pos + 1;
                            if (is_stop(p, t)) p.ctrl->halt = 1;
                        }
                    }
                }
            }
        }
        stamp();
        if (++ph == 5) {
            ph = 0;
            ++l;
        }
    }
    if (multi) {
        // Everything this CTA stored into the peers (logits rows, WKV state) must have landed before any
        // rank's kernel completes: fence, then a completion flag to CTA b of every rank, then wait for the
        // flags of the peers' CTA b.
        __threadfence_system();
        tok_sync();
        if (ctid == 0) {
            __threadfence_system();
            for (int g = 0; g < p.G; ++g)
                st_word(xch_at<unsigned long long>(p, g, p.off_done) + ((size_t)p.rank * nb + blockIdx.x), tag64(1u, p.tk), true);
        }
        if (ctid < 32) {
            const unsigned long long *d = xch_at<unsigned long long>(p, p.rank, p.off_done) + ((size_t)(ctid < p.G ? ctid : 0) * nb + blockIdx.x);
            unsigned long long a = 0;
            Waiter w = waiter_begin();
            for (;;) {
                bool bad = false;
                if (ctid < p.G) {
                    a = ld_word(d, true);
                    bad = (uint32_t)(a >> 32) != p.tk;
                }
                if (!__any_sync(0xffffffffu, bad)) break;
                if (waiter_tick(p, w)) wait_expired(p, kDiagDone, (unsigned int)p.L_run, (unsigned int)ctid, p.tk, (unsigned int)(a >> 32), 0ull);
            }
            __threadfence_system();
        }
    }
    // the sampler runs after the phase loop (the logits' row totals stay in shared memory) and is inlined: compiled as
    // a called function it gave the kernel local-memory traffic on the layer path (192-byte stack instead of 64) and
    // generate ran 11.6 % (1.5B) and 6.5 % (7B) slower per token than decode_timed; inlined, both run at the same
    // speed (profiles/r03_generate_breakdown.txt)
    if constexpr (GEN) {
        if (!p.greedy) sample_head(p, sm, sl.v0, sl.nv, ctid);
    }
    if (blockIdx.x == 0 && ctid == 0 && p.feed_mode == 2) p.ctrl->pos = p.ctrl->pos + 1;
    if ((p.dbg & 4) && p.trace != nullptr && ctid == 0)
        for (int i = 0; i < 16; ++i) p.trace[(size_t)blockIdx.x * kTraceMax + i] = (unsigned long long)sm.clk[i];
    stamp();
}

} // namespace rk
