// generate_kernels.cu — the token kernel's generate instantiations (k_token<CPL, FULL, false, true>), compiled as a
// translation unit of their own. The instantiations share the __noinline__ device functions of token_kernel.cuh
// (slice statistics, peer sums, the time-out path) with the other ones; in the same translation unit their extra
// call sites changed how ptxas scheduled the other instantiations, and the core loop's speed moves with its code
// generation (DESIGN.md section 9). Kept apart, engine.cu compiles the other instantiations exactly as before (the
// __noinline__ functions are `static` so that each translation unit has its own copy).
#include "token_kernel.cuh"

namespace rk {

const void *token_entry_gen(int cpl, bool full) {
#define X(A) \
    if (cpl == A) return full ? (const void *)k_token<A, true, false, true> : (const void *)k_token<A, false, false, true>;
    RK_CPLS(X)
#undef X
    return nullptr;
}

} // namespace rk
