#!/usr/bin/env python
"""bench.py — single-stream decode throughput of the B200 RWKV-v4 uint8 engine.

Contract (driver): `python bench.py --gpus N --steps K --warmup W [--impl reference]`
prints ONE JSON line on rank 0.

  step      one decoded token = ONE launch of the persistent token kernel (embedding .. head, + arg-max)
  workload  RWKV-4 7B shape (L=32, E=4096, uint8) — BASELINE.json's headline config — at every N (random-init
            weights written by tools/genmodel.cpp in the reference's .bin format); --workload 14b for config 5.
            N>1: ONE stream decoded by the N GPUs together (tensor parallel, strong scaling); N independent
            replicas are measured as well and reported under `alt`.
  value     tokens/s with everything resident in HBM: K launches back to back, each feeds the previous
            arg-max on the device; CUDA events on the engine stream, max over ranks.
  e2e       tokens/s through the C-ABI call a user makes (rwkv_b200_forward with HOST token and
            HOST logits buffer: 32 B H2D + 201,108 B D2H + host argmax every step).
  roofline  dominant kernel class: algorithmic bytes per launch / mean CUDA-event duration of
            that class, measured in this process by the engine's launch-by-launch profile run.
            Weights (7.2 GB) are >> L2 (126 MB), so every launch streams from HBM.
  cpu_baseline  the CPU oracle (port of the reference CUDA forward) on the host cores, a few
            tokens of the same model.
  --dump-outputs DIR   after the timed decode, what its last step computed, as a caller of the engine receives it:
            DIR/logits.npy (f32 [50277]) and DIR/state_{xy,aa,bb,pp,dd}.npy (f64 [L*E], the recurrent state the
            next token continues from; rank 0's copy when N > 1). The model and the token are seeded, so two
            builds run with the same arguments can be compared array by array.
  --impl reference   the UNMODIFIED reference CUDA build (oracle/_ref/ref_harness, compiled from
            /root/reference by oracle/Makefile) on GPU 0, same .bin, greedy decode through its
            own RWKV::forward, wall clock — the reference has no CPU forward (SURVEY.md 8c);
            its line also carries the oracle's cpu_baseline.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark runs from the tree build() left and writes nothing into it

SHAPES = {"169m": (12, 768), "1b5": (24, 2048), "7b": (32, 4096), "14b": (40, 5120)}
SEED = 20240924
SEED_TOKEN = 4118
VOCAB = 50277


def algorithmic_bytes_per_token(L, E):
    """BASELINE.md section 2: uint8 weights once per token + the small vector terms."""
    w = 13 * L * E * E + VOCAB * E
    return w + 4 * (20 * L * E + 2 * E) + 8 * (7 * L * E + 4 * (L + 1) * E) + 64 * L * E + 4 * E + 4 * VOCAB


def metric_name(workload):
    """BASELINE.json's metric; both arms print the identical string so that the driver can divide them."""
    return "tokens/sec single-stream decode RWKV-4 %s uint8; achieved HBM GB/s vs peak" % {"7b": "7B", "14b": "14B", "1b5": "1.5B", "169m": "169M"}[workload]


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu=0):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag, self.proc = gpu, [], False, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def model_path(workload, pkg):
    L, E = SHAPES[workload]
    base = os.environ.get("RWKV_B200_BENCH_DIR") or ("/dev/shm" if os.path.isdir("/dev/shm") else "/tmp")
    os.makedirs(base, exist_ok=True)
    path = os.path.join(base, "rwkv_b200_bench_%s_s%d.bin" % (workload, SEED))
    if not os.path.exists(path) or os.path.getsize(path) != pkg.build.file_bytes(L, E):
        tmp = path + ".tmp%d" % os.getpid()
        pkg.build.genmodel(L, E, SEED, tmp)
        os.replace(tmp, path)
    return path


def cpu_baseline(path, tokens, budget_s=25.0):
    """Oracle port on the host cores: a bounded sample of the same decode."""
    from oracle.oracle import Oracle
    orc = Oracle(path)
    n, t_total = 0, 0.0
    orc.forward(tokens[0])  # first token pages the mmap in; not timed
    for tok in tokens[1:]:
        t0 = time.perf_counter()
        orc.forward(tok)
        t_total += time.perf_counter() - t0
        n += 1
        if t_total > budget_s:
            break
    threads = orc.threads
    orc.close()
    return {"value": n / t_total if t_total > 0 else 0.0, "unit": "tokens/s", "cores": threads, "kind": "port",
            "sample": "%d tokens of the same model through oracle/rwkv_oracle.cpp (restatement of rwkv.cu), %d host threads" % (n, threads)}


def run_reference(args, pkg, workload):
    """--impl reference: the unmodified reference CUDA build on GPU 0."""
    from oracle.oracle import REF_HARNESS
    L, E = SHAPES[workload]
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base = {"impl": "reference", "metric": metric_name(workload), "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8 weights, f32/f64 math", "data": "synthetic",
            "config": {"workload": "RWKV-4 %s shape L=%d E=%d uint8, random-init, greedy single-stream decode" % (workload, L, E),
                       "l2": "weights >> L2, every token streams from HBM"}}
    if not os.path.exists(REF_HARNESS):
        base["unavailable"] = "oracle/_ref/ref_harness not built (needs /root/reference at build time)"
        emit(base)
        return
    path = model_path(workload, pkg)
    tf = path + ".seed.txt"
    with open(tf, "w") as f:
        f.write("%d\n" % SEED_TOKEN)
    dump = path + ".refdump"
    total = args.steps + args.warmup
    sampler = ClockSampler()
    sampler.start()
    r = subprocess.run([REF_HARNESS, path, tf, dump, "--warmup", str(args.warmup), "--dump-every", "0",
                        "--greedy", str(total)], capture_output=True, text=True)
    clocks = sampler.finish()
    res = None
    for line in r.stdout.splitlines():
        if line.startswith("REF_RESULT "):
            res = json.loads(line[len("REF_RESULT "):])
    if r.returncode != 0 or res is None:
        base["unavailable"] = "ref_harness failed rc=%d: %s" % (r.returncode, (r.stderr or r.stdout)[-300:].replace("\n", " "))
        emit(base)
        return
    toks = [int(x) for x in open(dump + ".tokens").read().split()][:6]
    cb = cpu_baseline(path, toks or [SEED_TOKEN] * 3, budget_s=20.0)
    v = res["tokens_per_s"]
    base.update({"value": v, "ms_per_step": 1000.0 / v if v else None, "clocks": clocks,
                 # the reference's forward copies the embedding row and the five state arrays up and the logits
                 # and the five state arrays down on every token (rwkv.h:353,372; rwkv.cu:467-490, 513-515)
                 "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 4 * E + 5 * L * E * 8,
                         "d2h_bytes_per_step": 4 * VOCAB + 5 * L * E * 8},
                 "cpu_baseline": cb, "gpu_launches": (9 + 20 * L) * args.steps,
                 "reference_arm": "unmodified /root/reference rwkv.cu + rwkv.h on 1 GPU (its own RWKV::forward incl. its host<->device state copies)"})
    for p in (dump, dump + ".tokens", tf):
        try:
            os.remove(p)
        except OSError:
            pass
    emit(base)


def ncu_traffic(kernel, workload):
    """DRAM bytes (read + write) per launch of the dominant kernel, from the committed `ncu --set full`
    capture of the same command (profiles/r02_token_traffic.json); null if there is none for this case."""
    p = os.path.join(ROOT, "profiles", "r02_token_traffic.json")
    try:
        with open(p) as f:
            t = json.load(f)
        if kernel == "token" and t.get("workload") == workload:
            return int(t["dram_bytes_read"]) + int(t["dram_bytes_write"])
    except (OSError, ValueError, KeyError):
        pass
    return None


def dump_outputs(out_dir, eng):
    """The last step's logits and the state after it, read back from the device after the timed region."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "logits.npy"), eng.debug_read("logits"))
    for k, v in eng.state_download().items():
        np.save(os.path.join(out_dir, "state_%s.npy" % k), v)


_REAL_STDOUT = None


def claim_stdout():
    """stdout carries exactly ONE JSON line: point fd 1 at stderr for everything libraries print (NCCL's version
    banner ignores NCCL_DEBUG_FILE) and keep the real stdout for emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    data = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(SHAPES))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the logits and the recurrent state of the last timed step as DIR/<name>.npy")
    ap.add_argument("--parallelism", default="tp", choices=["tp", "replicas"],
                    help="N > 1: which arrangement the headline `value` reports. 'tp' (default) = ONE stream decoded by the "
                         "N GPUs together (strong scaling: column/row split of every matrix, two in-kernel NVLink exchanges "
                         "per layer); 'replicas' = N independent streams, one per GPU (weak scaling, no exchange). The other "
                         "arrangement is measured too and reported under `alt`.")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    workload = args.workload or "7b"
    pkg = importlib.import_module("rwkv-cpp-accelerated_b200")

    if args.impl == "reference":
        run_reference(args, pkg, workload)
        return

    import numpy as np
    import torch
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    L, E = SHAPES[workload]
    if rank == 0:
        path = model_path(workload, pkg)
    if dist is not None:
        dist.barrier()
    path = model_path(workload, pkg)
    tp = world > 1 and args.parallelism == "tp"

    def make_engine(as_tp):
        if as_tp:
            e = pkg.Engine(path, device=local_rank, tp_rank=rank, tp_size=world)
            pkg.tp.connect(e)
            return e
        return pkg.Engine(path, device=local_rank)

    eng = make_engine(tp)

    # ---- warm-up (also builds the CUDA graphs) -------------------------------------------
    eng.state_zero()
    eng.decode_timed([SEED_TOKEN] * args.warmup, teacher_forced=False)

    def sync_all():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: device-resident greedy decode --------------------------------------------
    eng.state_zero()
    launches0 = eng.launch_count
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    sync_all()
    ms = eng.decode_timed([SEED_TOKEN] * args.steps, teacher_forced=False)
    sync_all()
    launches = eng.launch_count - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda:%d" % local_rank)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    tokens_total = args.steps if tp else args.steps * world  # tp: one stream over all GPUs; replicas: one per GPU
    value = tokens_total / (ms / 1e3)

    # ---- e2e: the user-facing call with host buffers -------------------------------------
    eng.state_zero()
    tok = SEED_TOKEN
    for _ in range(args.warmup):
        tok = int(eng.forward([tok])[0].argmax())
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        tok = int(eng.forward([tok])[0].argmax())
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda:%d" % local_rank)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = tokens_total / float(t.item())
    clocks = sampler.finish() if rank == 0 else None

    # ---- N > 1: also time the other arrangement of the same N GPUs ---------------------------------
    alt = None
    if world > 1:
        # never let the secondary measurement cost the headline line: every rank takes the same branch (a
        # failure to wire the peers is a property of the box, not of one rank), errors are reported in `alt`
        ok = torch.ones(1, device="cuda:%d" % local_rank)
        ms1, err = 0.0, None
        try:
            other = make_engine(not tp)
        except Exception as ex:  # noqa: BLE001
            other, err = None, str(ex)[:200]
            ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if float(ok.item()) > 0:
            other.decode_timed([SEED_TOKEN] * args.warmup, teacher_forced=False)
            other.state_zero()
            sync_all()
            ms1 = other.decode_timed([SEED_TOKEN] * args.steps, teacher_forced=False)
            sync_all()
        if other is not None:
            other.close()
        t = torch.tensor([ms1], dtype=torch.float64, device="cuda:%d" % local_rank)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        n_tok = args.steps * world if tp else args.steps
        alt = {"parallelism": ("replicas: %d independent streams, one per GPU (weak scaling)" % world) if tp
               else ("tp%d: ONE stream over %d GPUs (strong scaling; K/V/R/ffn-K/ffn-R/head split by output channel, "
                     "out-proj/ffn-V by input channel, two in-kernel NVLink exchanges of partial sums per layer, no NCCL "
                     "on the data path)" % (world, world))}
        if float(ok.item()) > 0:
            alt.update({"value": round(n_tok / (float(t.item()) / 1e3), 2), "unit": "tokens/s",
                        "ms_per_token_per_stream": round(float(t.item()) / args.steps, 5)})
        else:
            alt["error"] = err or "another rank could not set up this arrangement"

    def prof_run():
        eng.state_zero()
        toks = [SEED_TOKEN]
        tk = SEED_TOKEN
        for _ in range(7):
            tk = int(eng.forward([tk])[0].argmax())
            toks.append(tk)
        eng.state_zero()
        return toks, eng.profile(toks)

    if rank != 0:
        if tp:
            prof_run()  # every rank of a tensor-parallel group must launch what rank 0 launches
            dist.barrier()
        eng.close()
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- per-kernel roofline (launch-by-launch, CUDA events around every launch) ---------
    prof_tokens, prof = prof_run()
    if tp:
        dist.barrier()
    peak, peak_src = measured_peak()
    kernels = {}
    total_ms = sum(v["ms_sum"] for v in prof.values()) or 1.0
    for name, v in prof.items():
        if not v["launches"]:
            continue
        dur_ms = v["ms_sum"] / v["launches"]
        kernels[name] = {"launches_per_token": v["launches"] // len(prof_tokens), "us_per_launch": round(dur_ms * 1e3, 3),
                         "bytes_per_launch": int(v["bytes_per_launch"] / (world if tp else 1)),
                         "gbs": round(v["bytes_per_launch"] / (world if tp else 1) / dur_ms / 1e6, 1),
                         "share": round(v["ms_sum"] / total_ms, 4)}
    dom = max(kernels, key=lambda k: kernels[k]["share"])
    roofline = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["gbs"], "peak": peak, "unit": "GB/s",
                "frac": round(kernels[dom]["gbs"] / peak, 4), "traffic": ncu_traffic(dom, workload) if world == 1 else None, "peak_source": peak_src,
                "how": "algorithmic bytes per launch / mean CUDA-event duration per launch (eager profile run, %d tokens)" % len(prof_tokens)}
    abytes = algorithmic_bytes_per_token(L, E)
    if world > 1:
        # Launch-by-launch timing does not work across ranks (the peers' kernels of one token are not launched at the
        # same instant, so an eagerly timed launch mostly waits for them): take the timed decode itself - one launch
        # per token per GPU, CUDA events around the whole run, max over ranks - and the bytes ONE GPU streams per token.
        per_gpu = abytes * (value / world) / 1e9
        roofline.update({"achieved": round(per_gpu, 1), "frac": round(per_gpu / peak, 4),
                         "how": "algorithmic bytes one GPU streams per launch (%s) / (device-timed decode / launches), max over ranks"
                                % ("1/%d of a token's weights" % world if tp else "one token")})
    cb = None
    if not args.no_cpu_baseline and world == 1:
        cb = cpu_baseline(path, prof_tokens)
    eng.close()

    out = {
        "metric": metric_name(workload),
        "value": round(value, 2), "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms / args.steps, 5), "higher_is_better": True, "scaling": "strong" if tp else "weak", "vs_baseline": None,
        "dtype": "u8 weights x 23-bit fixed-point activations (byte limbs u8,u8,s8; exact int32 dp4a accumulate), f64 elementwise",
        "data": "synthetic",
        "config": {"workload": "RWKV-4 %s shape (L=%d, E=%d, V=50277) uint8, random-init reference-format .bin, greedy single-stream decode, batch 1" % (workload, L, E),
                   "l2": "inputs larger than L2: %.2f GB of weights per token vs 126 MB L2" % (abytes / 1e9),
                   "parallelism": ("tp%d: one stream; K/V/R/ffn-K/ffn-R/head split by output channel, out-proj/ffn-V by input "
                                   "channel, weights sharded at load, residual/layernorm replicated, two in-kernel exchanges of "
                                   "partial sums per layer as self-tagged words stored into the peers over NVLink (no NCCL on the "
                                   "data path)" % world) if tp
                   else ("replicas: 1 independent stream per GPU" if world > 1 else "1 GPU")},
        # per-GPU rate: tp -> each GPU streams 1/N of the bytes of every token; replicas -> 1/N of the tokens
        "hbm": {"algorithmic_bytes_per_token": abytes, "achieved_gbs": round(abytes * (value / world) / 1e9, 1),
                "frac_of_peak": round(abytes * (value / world) / 1e9 / peak, 4), "peak_gbs": peak, "peak_source": peak_src,
                "per": "GPU"},
        "roofline": roofline, "kernels": kernels,
        "e2e": {"value": round(e2e_value, 2), "unit": "tokens/s", "h2d_bytes_per_step": 32, "d2h_bytes_per_step": VOCAB * 4,
                "api": "rwkv_b200_forward(model, &token, 1, GPT, host_logits) + host argmax"},
        "gpu_launches": int(launches), "clocks": clocks, "cpu_baseline": cb,
    }
    if alt is not None:
        out["alt"] = alt
    emit(out)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
