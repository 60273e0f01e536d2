"""Regenerates tests/golden/reference/*.npz: greedy and teacher-forced runs of the UNMODIFIED reference CUDA build
(oracle/_ref/ref_harness, built by `make -C oracle ref` where the reference sources are present) on a B200, shrunk by
tests/util.py:shrink_reference_run to what tests/test_parity_gpu.py and tests/test_long_parity_gpu.py compare with.

  oracle_3x768                 3 x 768 synthetic model, teacher-forced on the CPU oracle's greedy stream, 8 tokens
  169m, 1b5, 7b, 14b           bench.py's models, greedy from token 4118: 256 / 1024 (every 4th step kept) / 64 / 64
  outliers, tiny_residual,     the 3 x 768 model with edited layernorms (tests/util.py:stress_model), teacher-forced
  offset_residual              on the oracle's greedy stream, 8 tokens

Run on the GPU:  python tests/golden/make_reference_golden.py [OUT_DIR]     (default: tests/golden/reference)
"""
import importlib
import os
import subprocess
import sys
import tempfile
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import bench  # noqa: E402
from oracle.oracle import REF_HARNESS, Oracle, read_ref_dump  # noqa: E402
from util import REFERENCE_GOLDEN, shrink_reference_run, stress_model  # noqa: E402

SEED = 20240924
SEED_TOKEN = 4118


def reference_run(path, td, tokens, greedy=0, dump_every=1):
    tf, dump = os.path.join(td, "toks.txt"), os.path.join(td, "ref.bin")
    with open(tf, "w") as f:
        f.write("\n".join(map(str, tokens)) + "\n")
    cmd = [REF_HARNESS, path, tf, dump, "--dump-every", str(dump_every)] + (["--greedy", str(greedy)] if greedy else [])
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("ref_harness failed:\n" + r.stdout[-2000:] + r.stderr[-2000:])
    d = read_ref_dump(dump)
    with open(dump + ".tokens") as f:
        fed = [int(x) for x in f.read().split()]
    os.remove(dump)
    return fed, d


def oracle_stream(path, n):
    orc = Oracle(path)
    toks, tok = [], SEED_TOKEN
    for _ in range(n):
        toks.append(tok)
        tok = int(orc.forward(tok).argmax())
    orc.close()
    return toks


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else REFERENCE_GOLDEN
    os.makedirs(out_dir, exist_ok=True)
    if not os.path.exists(REF_HARNESS):
        sys.exit("oracle/_ref/ref_harness not built")
    pkg = importlib.import_module("rwkv-cpp-accelerated_b200")
    pkg.build.build_all(force=False)

    def save(case, run):
        toks, d = run
        np.savez_compressed(os.path.join(out_dir, case + ".npz"),
                            **shrink_reference_run(toks, d["steps"], d["logits"], d["state"], zlib.crc32(case.encode())))
        print("%s: %d tokens, %d dumped steps" % (case, len(toks), len(d["steps"])), flush=True)

    with tempfile.TemporaryDirectory() as td:
        small = pkg.build.genmodel(3, 768, SEED, os.path.join(td, "syn_L3_E768.bin"))
        save("oracle_3x768", reference_run(small, td, oracle_stream(small, 8)))
        for kind in ("outliers", "tiny_residual", "offset_residual"):
            path = stress_model(small, os.path.join(td, "stress_%s.bin" % kind), kind)
            save(kind, reference_run(path, td, oracle_stream(path, 8)))
            os.remove(path)
        for workload, n, every in (("169m", 256, 1), ("1b5", 1024, 4), ("7b", 64, 1), ("14b", 64, 1)):
            save(workload, reference_run(bench.model_path(workload, pkg), td, [SEED_TOKEN], greedy=n, dump_every=every))


if __name__ == "__main__":
    main()
