"""Parity at the sizes and lengths BASELINE.json names, against the REFERENCE ITSELF (the unmodified
rwkv.cu + rwkv.h, run on a B200; its runs are stored under tests/golden/reference/ by
tests/golden/make_reference_golden.py): the reference decodes greedily, the engine replays the same tokens
teacher-forced, logits are compared step by step and the recurrent state at the end. Plus stress models for the
fixed-point activation quantiser and the layernorm statistics: outlier channels and a tiny or offset residual stream.

Tolerance (north_star): logits within 1e-3 of max|logits|; arg-max identical wherever the reference's own
top-1 / top-2 margin exceeds 1e-3 of max|logits|. A stored run keeps a sample of each logit vector and of the
state (tests/util.py:shrink_reference_run); the tolerance applies to every stored entry."""
import sys

import numpy as np
import pytest

from util import (ROOT, STATE_KEYS, load_reference, reference_logits_err, reference_margin, reference_state_err,
                  stress_model)

pytestmark = pytest.mark.gpu

REL_TOL = 1e-3
SEED_TOKEN = 4118


def rel_err(got, ref):
    return float(np.abs(got.astype(np.float64) - ref.astype(np.float64)).max() / max(np.abs(ref).max(), 1e-6))


def compare_with_reference(pkg, path, case, n_tokens, dump_every=1):
    ref = load_reference(case)
    toks = [int(t) for t in ref["tokens"]]
    assert len(toks) >= n_tokens
    want = {int(s): i for i, s in enumerate(ref["steps"])}
    assert all(s in want for s in range(0, n_tokens, dump_every))
    eng = pkg.Engine(path)
    worst, checked = 0.0, 0
    for step in range(n_tokens):
        if step in want:
            i = want[step]
            got = eng.forward([toks[step]])[0]
            e = reference_logits_err(got, ref, i)
            worst = max(worst, e)
            assert e < REL_TOL, "step %d: logits rel err %.3g" % (step, e)
            if reference_margin(ref, i) > 1e-3:
                assert int(got.argmax()) == int(ref["argmax"][i]), "step %d argmax" % step
                checked += 1
        else:
            eng.forward([toks[step]], want_logits=False)
    st = eng.state_download()
    for k in STATE_KEYS:
        assert reference_state_err(st[k], ref, k) < REL_TOL, "state %s" % k
    eng.close()
    return worst, checked, len(want)


def bench_model(pkg, workload):
    sys.path.insert(0, ROOT)
    import bench
    return bench.model_path(workload, pkg)


@pytest.mark.parametrize("workload,n_tokens,dump_every", [
    ("169m", 256, 1),    # BASELINE config 2: 169M storygen, 256 tokens
    ("1b5", 1024, 4),    # BASELINE config 3: 1.5B, 1k tokens
    ("7b", 64, 1),       # BASELINE config 4 (headline): the bench model itself
    ("14b", 64, 1),      # BASELINE config 5 at full depth (40 x 5120) on one GPU
])
def test_decode_matches_the_reference_at_baseline_sizes(pkg, workload, n_tokens, dump_every):
    worst, checked, compared = compare_with_reference(pkg, bench_model(pkg, workload), workload, n_tokens, dump_every)
    print("%s x %d tokens vs the reference CUDA build: worst logits rel err %.3g over %d compared steps, argmax checked on %d"
          % (workload, n_tokens, worst, compared, checked))


@pytest.mark.parametrize("kind", ["outliers", "tiny_residual", "offset_residual"])
def test_stress_models_match_oracle_and_reference(pkg, make_model, tmp_path, kind):
    """Activation vectors with outlier channels 10^2-10^3 x the median (real RWKV-4 checkpoints have them) leave
    the typical element few quantisation levels of the per-vector scale; a residual stream of magnitude 1e-3 or
    with |mean| >> std probes the layernorm statistics."""
    from oracle.oracle import Oracle
    path = stress_model(make_model(3, 768), str(tmp_path / ("stress_%s.bin" % kind)), kind)
    orc = Oracle(path)
    eng = pkg.Engine(path)
    toks, tok, worst = [], SEED_TOKEN, 0.0
    for step in range(8):
        toks.append(tok)
        got = eng.forward([tok])[0]
        ref = orc.forward(tok)
        assert np.all(np.isfinite(ref))
        e = rel_err(got, ref)
        worst = max(worst, e)
        assert e < REL_TOL, "%s step %d: logits rel err %.3g" % (kind, step, e)
        tok = int(ref.argmax())
    eng.close()
    orc.close()
    w2, _, _ = compare_with_reference(pkg, path, kind, 8)
    print("%s: worst logits rel err vs oracle %.3g, vs the reference CUDA build %.3g" % (kind, worst, w2))
