/* rwkv_b200.h — C ABI of the B200 (sm_100a) RWKV-v4 uint8 decode engine.
 *
 * This is the drop-in boundary: plain C, opaque handle, plain pointers and sizes,
 * no C++/torch types. Everything above it (include/rwkv/rwkv/rwkv.h, the pybind
 * module, bench.py via ctypes) is host glue; everything below it is hand-written
 * CUDA in rwkv-cpp-accelerated_b200/csrc/.
 *
 * Each entry point names the reference interface it replaces. Reference paths are
 * relative to harrisonvanderbyl/rwkv-cpp-accelerated:
 *   R.h  = include/rwkv/rwkv/rwkv.h      (backend hooks declared at R.h:63-122)
 *   R.cu = include/rwkv/cuda/rwkv.cu     (their CUDA implementation)
 *
 * Conventions: functions returning int return 0 on success and a non-zero code on
 * failure; rwkv_b200_last_error() then holds a message (thread-local). There is no
 * CPU fallback: without a usable sm_100 device every compute entry point fails.
 */
#ifndef RWKV_B200_H
#define RWKV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RWKV_B200_VOCAB 50277ULL
#define RWKV_B200_NUM_TENSORS 46

#define RWKV_B200_MODE_PARRALEL 0 /* enum MODE PARRALEL (include/rwkv/enums/enum.h:3) */
#define RWKV_B200_MODE_GPT 1      /* enum MODE GPT      (include/rwkv/enums/enum.h:4) */

typedef struct rwkv_b200_model rwkv_b200_model;

/* Last error message of the calling thread ("" if none). */
const char *rwkv_b200_last_error(void);

/* ABI version of this library (bumped on incompatible change). */
int rwkv_b200_abi_version(void);

/* Number of usable CUDA devices (0 if none / driver missing). Never throws. */
int rwkv_b200_device_count(void);

/* Load a reference-format model file onto `device` and repack it for decode.
 * Replaces `load(filename, ptrs, maxGPT)` (R.h:63, R.cu:638-717). The file layout is
 * 2 x int64 {n_layers, n_embed} followed by the 46 tensors in enum order
 * (converter/cpp_save_tensor.cpp:75-93). `max_gpt` is the number of state slots /
 * the longest token chunk a single forward may receive (R.h:281).
 * `quiet` = 0 prints the reference's "n_layers/n_embed/loading: <name>" lines.
 * Returns 0 and a handle in *out; non-zero if the file cannot be opened or parsed
 * (the reference calls exit(1) there, R.cu:641-645; the C++ wrapper keeps that). */
int rwkv_b200_load(const char *path, unsigned long long max_gpt, int device, int quiet,
                   rwkv_b200_model **out, unsigned long long *n_layers,
                   unsigned long long *n_embed);

/* Tensor-parallel load: this process is rank `tp_rank` of `tp_size` (1..8) ranks,
 * one GPU each, that decode ONE stream together (DESIGN.md section 7). Rank g owns the
 * att channels [g*E/G, (g+1)*E/G) and the ffn key channels [g*4E/G, ...): K, V, R, ffn-R,
 * ffn-K and the head are split by output channel, out-proj and ffn-V by input channel;
 * the loader reads and keeps only this rank's slices (1/G of every matrix; n_embed must
 * be a multiple of 16*G). The residual stream, layernorm and token shift are computed
 * identically on every rank; two in-kernel exchanges of partial sums per layer cross
 * NVLink. Every rank must make the same forward calls with the same tokens; all of them
 * receive the same logits and hold the complete recurrent state afterwards (state_download
 * works on any rank; state_upload must be given the same state on every rank).
 * `tp_size` = 1 is identical to rwkv_b200_load. After loading, wire the ranks with
 * rwkv_b200_tp_export / rwkv_b200_tp_import before the first forward. A rank that stops
 * calling makes the others fail with a time-out message (set_option "timeout_ms",
 * default 60000) instead of hanging. No reference counterpart (the reference is single-GPU). */
int rwkv_b200_load_tp(const char *path, unsigned long long max_gpt, int device, int quiet,
                      int tp_rank, int tp_size, rwkv_b200_model **out,
                      unsigned long long *n_layers, unsigned long long *n_embed);

/* Release every device and pinned-host allocation of the model.
 * Replaces `freeTensors(int**)` (R.h:77, R.cu:719-730). */
void rwkv_b200_free(rwkv_b200_model *m);

/* Device pointer that stands behind reference tensor-table slot `index`
 * (RWKV::tensors[index], R.h:249). State slots, scratch buffers and parameter
 * vectors keep the reference dtype and shape; the uint8 matrices are stored
 * repacked (row-major [out][in], value^0x80) — see DESIGN.md "HBM layout".
 * EMBED is a device pointer here (the reference keeps it on the host, R.cu:683). */
void *rwkv_b200_tensor(rwkv_b200_model *m, int index);

unsigned long long rwkv_b200_n_layers(const rwkv_b200_model *m);
unsigned long long rwkv_b200_n_embed(const rwkv_b200_model *m);
unsigned long long rwkv_b200_max_gpt(const rwkv_b200_model *m);

/* Pinned (page-locked) host memory for state mirrors / logits so copies are
 * asynchronous DMA. Falls back to malloc when no CUDA driver is present, so the
 * host API stays usable for tokenizer-only programs. */
void *rwkv_b200_host_alloc(size_t bytes);
void rwkv_b200_host_free(void *p);

/* Host -> device copy of the recurrent state, `slots` x n_layers x n_embed doubles per
 * array. Replaces `setState(...)` (R.h:64-66, R.cu:479-490). `pp` may be NULL
 * (the forward never reads or changes state_pp, R.cu:244,255). */
int rwkv_b200_state_upload(rwkv_b200_model *m, const double *xy, const double *aa,
                           const double *bb, const double *pp, const double *dd,
                           unsigned long long slots);

/* Device -> host copy of the recurrent state. Replaces the five state copies of
 * `getOutput(...)` (R.h:74-75, R.cu:472-476). NULL pointers are skipped. */
int rwkv_b200_state_download(rwkv_b200_model *m, double *xy, double *aa, double *bb,
                             double *pp, double *dd, unsigned long long slots);

/* Zero the device-resident state (what a fresh RWKVState holds, R.h:163-170). */
int rwkv_b200_state_zero(rwkv_b200_model *m);

/* One forward over `n_tokens` tokens on the device-resident state; blocks until the
 * logits are in `logits_out` (host, n_tokens x 50277 floats). One token = one launch of
 * the persistent token kernel; 8 tokens or more (one GPU; "prefill_min") run as int8
 * tensor-core GEMMs over the whole chunk with the weights streamed once per 128 tokens -
 * the same numbers; the chunk's launches are replayed as a CUDA graph per shape
 * (set_option "prefill" = "0" forces token by token, "prefill_graph" = "0" eager launches).
 * Replaces `cuda_rwkv_parralel(...)` + the logits copy of `getOutput`
 * (R.h:104-122, R.cu:493-593, 471). mode GPT: tokens are consumed in order on state
 * slot 0; mode PARRALEL: token t uses state slot t. n_tokens <= max_gpt.
 * `logits_out` may be NULL (state-only prefill: logits stay on the device). */
int rwkv_b200_forward(rwkv_b200_model *m, const unsigned long long *tokens,
                      unsigned long long n_tokens, int mode, float *logits_out);

/* Same as rwkv_b200_forward(.., 1 token, GPT) followed by an on-device argmax;
 * returns the arg-max token in *next. Used by greedy decode loops so only 8 bytes
 * cross PCIe per token. `logits_out` may be NULL. */
int rwkv_b200_forward_greedy(rwkv_b200_model *m, unsigned long long token,
                             unsigned long long *next, float *logits_out);

/* Pinned host buffer (max_gpt x 50277 floats) the engine copies logits into; passing
 * it as `logits_out` avoids one host-side memcpy. This is what RWKV::out points at. */
float *rwkv_b200_logits_host(rwkv_b200_model *m);

/* Test hook: copy a named device vector ("x" = residual stream after the last layer,
 * "logits", "trace", "ptrace") to `dst`. Returns the element count, or -1. */
long long rwkv_b200_debug_read(rwkv_b200_model *m, const char *name, void *dst, size_t dst_bytes);

/* --- measurement hooks (bench.py); not part of the reference surface ------------ */

/* Decode `n` tokens taken from `tokens` (host array, copied to HBM before timing) on
 * the resident state with no host<->device traffic inside the timed region; CUDA
 * events on the engine's stream bracket the whole run. Returns elapsed ms in *ms.
 * If `teacher_forced` is 0 only tokens[0] is used and each next token is the
 * on-device argmax of the previous logits. */
int rwkv_b200_decode_timed(rwkv_b200_model *m, const unsigned long long *tokens,
                           unsigned long long n, int teacher_forced, float *ms);

/* Number of distinct kernels in one single-token forward (1: the token kernel), and their names. */
int rwkv_b200_kernel_count(void);
const char *rwkv_b200_kernel_name(int k);

/* Run `n` single-token forwards with a CUDA-event pair around every launch.
 * ms_sum[k] = total ms spent in kernel class k, launches[k] = launch count,
 * bytes[k] = algorithmic HBM bytes of ONE launch of class k on this rank (its share of the
 * weights + the vectors). */
int rwkv_b200_profile(rwkv_b200_model *m, const unsigned long long *tokens,
                      unsigned long long n, float *ms_sum, unsigned long long *launches,
                      double *bytes);

/* Kernel launches issued by this model since load (for bench.py "gpu_launches"). */
unsigned long long rwkv_b200_launch_count(const rwkv_b200_model *m);

/* Device-side restatement of `typical(logits, temp, tau)` (R sampler/typical.h:20-58 as it actually
 * behaves, see include/rwkv/sampler/typical.h) on the logits of the LAST forward, which never leave
 * the GPU: probs = exp(l)/sum, probs ^ uint8(1/temp), cumulative sums, first index whose cumulative
 * probability reaches `u`, the uniform in [0,1) the caller drew from its generator
 * (std::generate_canonical<double,53> keeps the reference's random stream). `*margin` is the distance
 * of `u` to the nearest interval boundary; device sums are block reductions, so a caller that wants
 * the host's token in every case re-samples on the host when margin < 1e-9 (RWKV::sample does). */
int rwkv_b200_sample_typical(rwkv_b200_model *m, float temp, double u, unsigned long long *token,
                             double *margin);

/* Free-running generation on state slot 0: exactly `n` iterations of
 *     logits = forward(tok); tok = pick(logits)
 * starting from `first_token`, as back-to-back launches of the token kernel that pick the
 * next token on the device (no host round trip per token). pick is
 *   RWKV_B200_GEN_GREEDY : the arg-max (first index of the largest logit);
 *   RWKV_B200_GEN_TYPICAL: typical_with_u(logits, temp, uniforms[i]) of
 *                          include/rwkv/sampler/typical.h, i.e. exactly what
 *                          rwkv_sampler_pick returns on the host for that uniform. The device
 *                          sums differ from the host's sequential ones by ~1e-13, so a step
 *                          whose uniform lies closer than set_option "sample_margin" (default
 *                          1e-9) to an interval boundary is finished on the host with the same
 *                          uniform: the result is always the host sampler's token stream.
 * `uniforms`: n values in [0, 1) (TYPICAL only; may be NULL for GREEDY), one per step, e.g.
 * std::generate_canonical<double, 53> draws of the caller's generator. `temp` > 1/256.
 * `stop`: up to 8 token ids; the run ends after the first step that produces one of them.
 * After the call the state has consumed first_token, t1, ..., t(k-1); tokens_out[0..k) =
 * t1..tk with k = *n_out, and k < n only if tk is a stop id. The device logits, and
 * `logits_out` (50277 floats) if not NULL, are those of the last forward, so
 * rwkv_b200_sample_typical and rwkv_b200_logits_host stay consistent with it.
 * Errors (no device work done): tensor parallelism (tp_size > 1 is not supported), a token
 * or stop id >= vocabulary, a uniform outside [0, 1), n == 0, a NULL output.
 * No reference counterpart (the reference samples on the host after every forward). */
#define RWKV_B200_GEN_GREEDY 0
#define RWKV_B200_GEN_TYPICAL 1
int rwkv_b200_generate(rwkv_b200_model *m, unsigned long long first_token, unsigned long long n,
                       int how, float temp, const double *uniforms,
                       const unsigned long long *stop, int n_stop,
                       unsigned long long *tokens_out, unsigned long long *n_out,
                       float *logits_out);

/* Engine knobs (all optional), key/value strings: "window" / "bwindow" (bulk copies in
 * flight per SM while streaming / while the CTAs exchange vectors), "pf_dist" (tiles the L2
 * prefetch runs ahead), "stages" (ring depth), "poll_first", "timeout_ms", "max_layers",
 * "trace", "prefill", "prefill_min", "prefill_graph", "grid" (CTAs, at most the SM count),
 * "cluster" (1, 2 or 4 CTAs share a gather through distributed shared memory; measured
 * without gain, default 1), "sample_margin" (rwkv_b200_generate: smallest distance of a
 * uniform to an interval boundary the device's sampled token is kept at, in [0, 1], default
 * 1e-9). Returns non-zero for an unknown key. */
int rwkv_b200_set_option(rwkv_b200_model *m, const char *key, const char *value);

/* --- tensor-parallel wiring (tp_size > 1 only) --------------------------------- */

/* Size in bytes of this rank's peer-visible exchange block (tagged activation vectors,
 * per-CTA records, inboxes of the cross-GPU partial sums, logits, WKV state); allocated by
 * the load. */
size_t rwkv_b200_tp_buffer_bytes(const rwkv_b200_model *m);
/* Export this rank's exchange buffer as a CUDA IPC handle (64 bytes). */
int rwkv_b200_tp_export(rwkv_b200_model *m, void *ipc_handle_64);
/* Import every rank's handle (tp_size x 64 bytes, own rank's entry ignored). */
int rwkv_b200_tp_import(rwkv_b200_model *m, const void *ipc_handles);

#ifdef __cplusplus
}
#endif
#endif /* RWKV_B200_H */
