import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INCLUDE = os.path.join(ROOT, "include")
PKG_DIR = os.path.join(ROOT, "rwkv-cpp-accelerated_b200")
VOCAB_DIR = os.path.join(INCLUDE, "rwkv", "tokenizer", "vocab")
REFERENCE_GOLDEN = os.path.join(ROOT, "tests", "golden", "reference")
VOCAB = 50277
STATE_KEYS = ("xy", "aa", "bb", "dd")


def compile_cpp(src, out, link_engine=False, extra=()):
    cmd = ["g++", "-O1", "-std=c++17", "-I" + INCLUDE, src, "-o", out] + list(extra)
    if link_engine:
        cmd += ["-L" + PKG_DIR, "-lrwkv_b200", "-Wl,-rpath," + PKG_DIR]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, "g++ failed:\n" + r.stderr[-4000:]
    return out


def stress_model(src, dst, kind, L=3, E=768):
    """A copy of the synthetic L x E model `src` with its layernorm parameters edited in place.
    LAYERNORMS = f64 [4(L+1)][E] after xbuf (f64 [E]) and embed (f32 [V][E]): rows 0,1 = ln0 w,b;
    4i+2, 4i+3 = ln1 of layer i; 4(i+1), 4(i+1)+1 = ln2 of layer i (convert_model.py:30-46)."""
    import shutil
    shutil.copyfile(src, dst)
    ln = np.memmap(dst, dtype=np.float64, mode="r+", offset=16 + 8 * E + 4 * VOCAB * E, shape=(4 * (L + 1), E))
    if kind == "outliers":
        rng = np.random.default_rng(7)
        for i in range(L):
            ch = rng.choice(E, size=3, replace=False)
            ln[4 * i + 2, ch] *= 300.0      # ln1 weight: three channels 300x the rest
            ln[4 * (i + 1), ch] *= 300.0    # ln2 weight
    elif kind == "tiny_residual":
        ln[0] *= 1e-3                       # ln0 weight and bias: residual stream of magnitude 1e-3
        ln[1] *= 1e-3
    elif kind == "offset_residual":
        ln[1] += 50.0                       # ln0 bias: |mean| >> std in every later layernorm
    else:
        raise ValueError(kind)
    ln.flush()
    del ln
    return dst


# ---- stored runs of the reference CUDA build (tests/golden/make_reference_golden.py) --------------------------------
# A full run (50277 logits per step, the whole f64 state) is megabytes; what is kept is enough to apply the parity
# tolerances: per dumped step the arg-max, the two largest logits, max|logits| and the logits at a fixed seeded sample
# of the vocabulary; of the final state max|.| and the values at a seeded sample of positions that includes the
# position of max|.|.
LOGIT_SAMPLE = 32
STATE_SAMPLE = 64


def shrink_reference_run(tokens, steps, logits, state, seed):
    rng = np.random.default_rng(seed)
    lg = np.stack(logits).astype(np.float32)
    vidx = np.sort(rng.choice(lg.shape[1], LOGIT_SAMPLE, replace=False))
    top = np.sort(np.partition(lg, -2, axis=1)[:, -2:], axis=1)[:, ::-1]
    out = {"tokens": np.asarray(tokens, np.int64), "steps": np.asarray(steps, np.int64), "vocab_idx": vidx.astype(np.int64),
           "logits": lg[:, vidx], "argmax": lg.argmax(axis=1).astype(np.int64), "top2": np.ascontiguousarray(top),
           "absmax": np.abs(lg).max(axis=1)}
    for k in STATE_KEYS:
        s = np.asarray(state[k], np.float64)
        idx = np.unique(np.append(rng.choice(s.size, STATE_SAMPLE, replace=False), np.abs(s).argmax()))
        out["state_%s_idx" % k] = idx.astype(np.int64)
        out["state_%s" % k] = s[idx]
        out["state_%s_absmax" % k] = np.float64(np.abs(s).max())
    return out


def load_reference(case):
    with np.load(os.path.join(REFERENCE_GOLDEN, case + ".npz")) as z:
        return {k: z[k] for k in z.files}


def reference_logits_err(got, ref, i):
    """max |got - reference| / max|reference logits| of dumped step i, over the stored entries (the vocabulary sample
    and the reference's arg-max) and max|logits| itself."""
    got = np.asarray(got, np.float64)
    d = max(float(np.abs(got[ref["vocab_idx"]] - ref["logits"][i]).max()),
            abs(float(got[ref["argmax"][i]]) - float(ref["top2"][i, 0])),
            abs(float(np.abs(got).max()) - float(ref["absmax"][i])))
    return d / max(float(ref["absmax"][i]), 1e-6)


def reference_margin(ref, i):
    """The reference's own top-1 / top-2 margin at dumped step i, relative to max|logits|."""
    return float((ref["top2"][i, 0] - ref["top2"][i, 1]) / max(float(ref["absmax"][i]), 1e-6))


def reference_state_err(st, ref, k):
    idx = ref["state_%s_idx" % k]
    return float(np.abs(np.asarray(st)[idx] - ref["state_%s" % k]).max() / max(float(ref["state_%s_absmax" % k]), 1e-6))
