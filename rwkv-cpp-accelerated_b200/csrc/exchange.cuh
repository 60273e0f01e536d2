// exchange.cuh — how CTAs (and GPUs) hand small vectors to each other inside the token kernel.
//
// There is no grid barrier and no atomic on the data path. Every exchanged word carries its own
// sequence tag, so a reader simply polls the data it needs until the tag says "this epoch":
//
//   * 8-byte words {payload32, tag32}: partial sums (a double travels as two such words), sigmoid
//     values, arg-max candidates, completion flags. tag = epoch (never 0; buffers start zeroed).
//   * 4-byte words for the activation vectors that feed a GEMV: an f32 whose two low mantissa bits
//     are the tag (epoch & 3). The value is rounded to 22 mantissa bits by the writer, which is the
//     resolution of the 23-bit limb quantiser that consumes it anyway.
//
// Aligned 4- and 8-byte accesses are single-copy atomic, vector accesses are performed element-wise,
// so a reader can never observe a payload that does not belong to the tag it sees; no fence, no
// release/acquire pair, no round trip before the flag (the cost a barrier cannot avoid). A word is
// rewritten one epoch later by the same writer, and every exchange is all-to-all (each output of
// phase n depends on every output of phase n-1), so a writer cannot run ahead far enough to overwrite
// a word a reader still needs; the previous content always carries the previous tag.
//
// Across GPUs the same words are stored straight into the peer's exchange block over NVLink
// (st.relaxed.sys to the peer-mapped address); every read is local.
#pragma once
#include "common.cuh"

namespace rk {

struct __align__(16) TaggedDouble { unsigned long long w[2]; }; // {lo32 | tag, hi32 | tag}

__device__ __forceinline__ unsigned long long tag64(uint32_t payload, uint32_t tag) {
    return ((unsigned long long)tag << 32) | (unsigned long long)payload;
}

// ---- stores -------------------------------------------------------------------------------------
__device__ __forceinline__ void st_pair(void *p, unsigned long long a, unsigned long long b, bool sys) {
    if (sys) asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(a), "l"(b) : "memory");
    else asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}
__device__ __forceinline__ void st_word(void *p, unsigned long long a, bool sys) {
    if (sys) asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(a) : "memory");
    else asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(a) : "memory");
}
__device__ __forceinline__ void st_tagged_double(void *p, double v, uint32_t tag, bool sys) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(v);
    st_pair(p, tag64((uint32_t)u, tag), tag64((uint32_t)(u >> 32), tag), sys);
}
__device__ __forceinline__ void st_f32(float *p, uint32_t bits) {
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(bits) : "memory");
}
// f32 with the tag in its two low mantissa bits (value rounded to nearest at that resolution)
__device__ __forceinline__ uint32_t tag_f32(float v, uint32_t tag2) { return ((__float_as_uint(v) + 2u) & ~3u) | tag2; }
__device__ __forceinline__ float untag_f32(uint32_t bits) { return __uint_as_float(bits & ~3u); }

// ---- loads --------------------------------------------------------------------------------------
__device__ __forceinline__ void ld_pair(const void *p, unsigned long long &a, unsigned long long &b, bool sys) {
    if (sys) asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
    else asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ unsigned long long ld_word(const void *p, bool sys) {
    unsigned long long a;
    if (sys) asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(a) : "l"(p) : "memory");
    else asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(a) : "l"(p) : "memory");
    return a;
}
__device__ __forceinline__ uint4 ld_vec4(const void *p) {
    uint4 v;
    asm volatile("ld.relaxed.gpu.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ bool tags_ok(unsigned long long a, unsigned long long b, uint32_t tag) {
    return (uint32_t)(a >> 32) == tag && (uint32_t)(b >> 32) == tag;
}
__device__ __forceinline__ double pair_to_double(unsigned long long a, unsigned long long b) {
    return __longlong_as_double((long long)(((b & 0xffffffffull) << 32) | (a & 0xffffffffull)));
}
__device__ __forceinline__ bool vec4_ok(const uint4 &v, uint32_t tag2) {
    // all four low-2-bit fields equal tag2
    return (((v.x ^ tag2) | (v.y ^ tag2) | (v.z ^ tag2) | (v.w ^ tag2)) & 3u) == 0u;
}

// ---- bounded waiting ------------------------------------------------------------------------------
// A wait that does not complete within Params::timeout_ms writes a Diag record to mapped host memory
// and traps: a protocol bug or a peer rank that never launched becomes an error message instead of a hang.
struct Waiter {
    unsigned long long deadline;
    unsigned int spins;
};
__device__ __forceinline__ Waiter waiter_begin() { return Waiter{0ull, 0u}; }
static __device__ __noinline__ void wait_expired(const Params &p, unsigned int code, unsigned int layer, unsigned int kind,
                                          unsigned int expect, unsigned int seen, unsigned long long aux) {
    Diag *d = p.diag;
    if (d != nullptr && atomicCAS(&d->code, 0u, code) == 0u) {
        d->rank = (unsigned int)p.rank;
        d->cta = blockIdx.x;
        d->thread = threadIdx.x;
        d->layer = layer;
        d->kind = kind;
        d->expect = expect;
        d->seen = seen;
        d->aux = aux;
        __threadfence_system();
    }
    __trap();
}
// Call once per failed poll. Returns true when the wait has expired.
__device__ __forceinline__ bool waiter_tick(const Params &p, Waiter &w) {
    if ((++w.spins & 1023u) != 0u) return false;
    const unsigned long long now = globaltimer();
    if (w.deadline == 0ull) {
        w.deadline = now + (unsigned long long)p.timeout_ms * 1000000ull;
        return false;
    }
    return now > w.deadline;
}

__device__ __forceinline__ void mbar_wait(const Params &p, uint32_t bar, uint32_t parity, unsigned int code) {
    Waiter w = waiter_begin();
    while (!mbar_try_wait(bar, parity)) {
        if (waiter_tick(p, w)) wait_expired(p, code, 0, 0, parity, 0, bar);
    }
}

template <class T> __device__ __forceinline__ T *xch_at(const Params &p, int g, unsigned long long off) {
    return reinterpret_cast<T *>(p.xch[g] + off);
}

} // namespace rk
