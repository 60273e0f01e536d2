"""Per-token time of each decode path at the 169M / 1.5B / 7B shapes, whole model and head only (max_layers=0), to
see where generate's time goes: decode_timed (bench.py's greedy kernel, CUDA events), generate GREEDY / TYPICAL
(exponents 1 and 3), forward with and without the logits copy, and the one-CTA sample_typical call alone.
Wall time over 256 tokens, median of 3 after a warm-up. usage: python generate_breakdown.py"""
import importlib
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

pkg = importlib.import_module("rwkv-cpp-accelerated_b200")
N = 256
G, T = pkg.engine.GEN_GREEDY, pkg.engine.GEN_TYPICAL


def per_token_us(fn, reps=3):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return 1e6 * float(np.median(ts)) / N


for shape in ("169m", "1b5", "7b"):
    eng = pkg.Engine(bench.model_path(shape, pkg))
    us = np.random.default_rng(1).random(N)
    tok = bench.SEED_TOKEN
    for ml in (-1, 0):
        eng.set_option("max_layers", ml)
        eng.state_zero()
        g = per_token_us(lambda: eng.generate(tok, N, G, 1.0, None, want_logits=False))
        t1 = per_token_us(lambda: eng.generate(tok, N, T, 0.9, us, want_logits=False))
        t3 = per_token_us(lambda: eng.generate(tok, N, T, 0.3, us, want_logits=False))
        dev = eng.decode_timed([tok] * N, teacher_forced=False) * 1e3 / N
        fw = per_token_us(lambda: [eng.forward([tok]) for _ in range(N)])
        fwn = per_token_us(lambda: [eng.forward([tok], want_logits=False) for _ in range(N)])
        st = per_token_us(lambda: [eng.sample_typical(0.9, 0.5) for _ in range(N)])
        print("%s max_layers=%d us/token: decode_timed %.1f gen_greedy %.1f gen_typical(e=1) %.1f gen_typical(e=3) %.1f "
              "forward+logits %.1f forward-no-logits %.1f sample_typical %.1f" % (shape, ml, dev, g, t1, t3, fw, fwn, st), flush=True)
    eng.close()
