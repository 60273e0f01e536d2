"""Sampled vs greedy free-running generation against the per-token host loop, at the 169M / 1.5B / 7B shapes
(synthetic models of bench.py). For each shape, from the same state and the same seeded uniforms:

  loop     forward(token) -> logits to the host, then sample_typical(temp, u) (host sampler when its margin < 1e-9):
           the two calls and two synchronisations per token that RWKV::forward + RWKV::sample make
  typical  rwkv_b200_generate(TYPICAL): the sampler runs inside the token kernel, one synchronisation per call
  greedy   rwkv_b200_generate(GREEDY): the on-device arg-max, the same launches as bench.py's decode

tokens/s = steps / wall time of the call(s), which end in a device synchronisation; median of --repeats runs after
one warm-up run. The three token streams are checked against a host recomputation: the loop's and generate's
sampled tokens against the numpy restatement of the sampler on the loop's logits, the greedy tokens against
forward + arg-max. The device name and power limit are read in the same process.
usage: python generate_bench.py [--steps 128] [--repeats 3] [--temp 0.9] [--shapes 169m,1b5,7b] [--out FILE]"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

pkg = importlib.import_module("rwkv-cpp-accelerated_b200")


def host_pick(logits, temp, u):
    """include/rwkv/sampler/typical.h restated in numpy (float64, sequential cumulative sum)."""
    p = np.exp(logits.astype(np.float64))
    p /= p.sum()
    e = int(np.uint8(int(1.0 / temp))) if temp != 1.0 else 1
    p = np.ones_like(p) if e == 0 else p ** e
    cp = np.cumsum(p / p.sum())
    cp[-1] = 1.0
    return int(np.searchsorted(cp, u, side="left"))


def device_info():
    q = "name,power.limit,clocks.max.sm,driver_version"
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power, clk, drv = [x.strip() for x in r.stdout.strip().split(",")]
        return {"device": name, "power_limit": power, "sm_max_clock": clk, "driver": drv}
    except Exception as ex:  # noqa: BLE001
        return {"device": "unknown (%s)" % ex}


def run_loop(eng, steps, temp, us):
    toks, logits, tok = [], [], bench.SEED_TOKEN
    t0 = time.perf_counter()
    for i in range(steps):
        lg = eng.forward([tok])[0]
        tok, margin = eng.sample_typical(temp, float(us[i]))
        if margin < 1e-9:  # what RWKV::sample does: the host decides
            tok = host_pick(lg, temp, us[i])
        toks.append(tok)
        logits.append(lg)
    return time.perf_counter() - t0, toks, logits


def run_generate(eng, steps, how, temp, us):
    t0 = time.perf_counter()
    toks, _ = eng.generate(bench.SEED_TOKEN, steps, how, temp, us, want_logits=False)
    return time.perf_counter() - t0, toks


def measure(shape, steps, repeats, temp):
    eng = pkg.Engine(bench.model_path(shape, pkg))
    us = np.random.default_rng(20240924).random(steps)
    res = {}
    for name in ("loop", "typical", "greedy"):
        times = []
        for r in range(repeats + 1):  # run 0 warms up
            eng.state_zero()
            if name == "loop":
                dt, toks, logits = run_loop(eng, steps, temp, us)
                loop_toks, loop_logits = toks, logits
            elif name == "typical":
                dt, toks = run_generate(eng, steps, pkg.engine.GEN_TYPICAL, temp, us)
                typ_toks = toks
            else:
                dt, toks = run_generate(eng, steps, pkg.engine.GEN_GREEDY, temp, None)
                greedy_toks = toks
            if r > 0:
                times.append(dt)
        t = float(np.median(times))
        res[name] = {"tok_s": round(steps / t, 1), "ms_per_token": round(1e3 * t / steps, 4),
                     "runs_s": [round(x, 5) for x in times]}
    # host recomputation of the three streams
    host = [host_pick(lg, temp, u) for lg, u in zip(loop_logits, us)]
    assert loop_toks == host, "%s: forward + sample_typical differs from the host sampler" % shape
    assert typ_toks == host, "%s: generate(TYPICAL) differs from the host sampler" % shape
    eng.state_zero()
    ref, tok = [], bench.SEED_TOKEN
    for _ in range(steps):
        tok = int(eng.forward([tok])[0].argmax())
        ref.append(tok)
    assert greedy_toks == ref, "%s: generate(GREEDY) differs from forward + argmax" % shape
    eng.close()
    L, E = bench.SHAPES[shape]
    return {"shape": shape, "L": L, "E": E, "steps": steps, "repeats": repeats, "temp": temp, "streams_checked": True,
            **res, "typical_vs_greedy": round(res["typical"]["tok_s"] / res["greedy"]["tok_s"], 4),
            "typical_vs_loop": round(res["typical"]["tok_s"] / res["loop"]["tok_s"], 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--temp", type=float, default=0.9)
    ap.add_argument("--shapes", default="169m,1b5,7b")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    info = device_info()
    rows = [measure(s, a.steps, a.repeats, a.temp) for s in a.shapes.split(",")]
    lines = ["device: %s, power limit %s, max SM clock %s, driver %s" % (info.get("device"), info.get("power_limit"),
                                                                          info.get("sm_max_clock"), info.get("driver")),
             "", "| shape | loop tok/s | generate TYPICAL tok/s | generate GREEDY tok/s | TYPICAL / GREEDY | TYPICAL / loop |",
             "|---|---|---|---|---|---|"]
    for r in rows:
        lines.append("| %s (L=%d, E=%d) | %.1f | %.1f | %.1f | %.3f | %.3f |" % (
            r["shape"], r["L"], r["E"], r["loop"]["tok_s"], r["typical"]["tok_s"], r["greedy"]["tok_s"],
            r["typical_vs_greedy"], r["typical_vs_loop"]))
    text = "\n".join(lines) + "\n\n" + "\n".join(json.dumps({**info, **r}) for r in rows) + "\n"
    print(text, end="")
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
