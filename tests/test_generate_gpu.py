"""rwkv_b200_generate: free-running generation with the next token picked inside the token kernel (arg-max or the
typical sampler). The reference for every check is the same engine driven one token at a time; the engine is
bit-deterministic, so "identical" means identical."""
import os
import subprocess

import numpy as np
import pytest

from util import ROOT, STATE_KEYS, compile_cpp

pytestmark = pytest.mark.gpu

SEED_TOKEN = 4118


def host_pick(logits, temp, u):
    """include/rwkv/sampler/typical.h restated in numpy (float64, sequential cumulative sum)."""
    p = np.exp(logits.astype(np.float64))
    p /= p.sum()
    e = int(np.uint8(int(1.0 / temp))) if temp != 1.0 else 1
    p = np.ones_like(p) if e == 0 else p ** e
    cp = np.cumsum(p / p.sum())
    cp[-1] = 1.0
    return int(np.searchsorted(cp, u, side="left"))


def loop(eng, first, n, temp=None, us=None, stop=()):
    """forward + pick, one token per call: (tokens t1..tk, logits of the last forward)."""
    toks, tok, logits = [], first, None
    for i in range(n):
        logits = eng.forward([tok])[0]
        tok = int(logits.argmax()) if temp is None else host_pick(logits, temp, us[i])
        toks.append(tok)
        if tok in stop:
            break
    return toks, logits


def assert_same_state(eng, ref_state):
    sa, sb = eng.state_download(), ref_state
    for k in STATE_KEYS:
        assert np.array_equal(sa[k], sb[k]), "state %s differs" % k


def uniforms(n, seed):
    return np.random.default_rng(seed).random(n)


@pytest.mark.parametrize("E", [768, 2048, 4096, 5120])
def test_greedy_matches_forward_argmax(pkg, make_model, E):
    eng = pkg.Engine(make_model(2, E))
    ref_toks, ref_logits = loop(eng, SEED_TOKEN, 16)
    ref_state = eng.state_download()
    eng.state_zero()
    toks, logits = eng.generate(SEED_TOKEN, 16, pkg.engine.GEN_GREEDY)
    assert toks == ref_toks
    assert np.array_equal(logits, ref_logits)
    assert np.array_equal(eng.debug_read("logits"), ref_logits)
    assert_same_state(eng, ref_state)
    eng.close()


@pytest.mark.parametrize("temp", [0.9, 0.5, 0.3, 2.0])  # exponents 1, 2, 3, 0
def test_typical_matches_host_sampler(pkg, make_model, temp):
    eng = pkg.Engine(make_model(2, 768))
    us = uniforms(64, 11)
    ref_toks, ref_logits = loop(eng, SEED_TOKEN, 64, temp, us)
    ref_state = eng.state_download()
    eng.state_zero()
    toks, logits = eng.generate(SEED_TOKEN, 64, pkg.engine.GEN_TYPICAL, temp, us)
    assert toks == ref_toks
    assert np.array_equal(logits, ref_logits)
    assert_same_state(eng, ref_state)
    eng.close()


def median_margin(eng, first, n, temp, us):
    """The device sampler's margins along the reference run (logits of each step)."""
    margins, tok = [], first
    for i in range(n):
        logits = eng.forward([tok])[0]
        margins.append(eng.sample_typical(temp, float(us[i]))[1])
        tok = host_pick(logits, temp, us[i])
    return float(np.median(margins))


@pytest.mark.parametrize("threshold", ["1", "median"])
def test_host_fallback_keeps_the_host_stream(pkg, make_model, threshold):
    eng = pkg.Engine(make_model(2, 768))
    temp, us = 0.9, uniforms(48, 5)
    if threshold == "median":  # about half the steps halt, the others run free between them
        threshold = repr(median_margin(eng, SEED_TOKEN, 48, temp, us))
        eng.state_zero()
    ref_toks, ref_logits = loop(eng, SEED_TOKEN, 48, temp, us)
    ref_state = eng.state_download()
    eng.state_zero()
    eng.set_option("sample_margin", threshold)
    toks, logits = eng.generate(SEED_TOKEN, 48, pkg.engine.GEN_TYPICAL, temp, us)
    assert toks == ref_toks
    assert np.array_equal(logits, ref_logits)
    assert_same_state(eng, ref_state)
    eng.close()


@pytest.mark.parametrize("L", [1, 3, 5, 6])  # L + 1 = 2, 4, 6, 7: every residue mod 4 of a launch's epoch advance
def test_epochs_after_halted_launches(pkg, make_model, L):
    path = make_model(L, 768)
    eng, fresh = pkg.Engine(path), pkg.Engine(path)
    temp, us = 0.9, uniforms(40, 3 + L)
    eng.set_option("sample_margin", repr(median_margin(eng, SEED_TOKEN, 40, temp, us)))
    eng.state_zero()
    toks, _ = eng.generate(SEED_TOKEN, 40, pkg.engine.GEN_TYPICAL, temp, us)
    ref_toks, _ = loop(fresh, SEED_TOKEN, 40, temp, us)
    assert toks == ref_toks
    # after the halts: single forwards, then more generation, on both engines
    for t in (toks[-1], 17, 50000):
        assert np.array_equal(eng.forward([t])[0], fresh.forward([t])[0])
    more, lg = eng.generate(123, 12, pkg.engine.GEN_GREEDY)
    ref_more, ref_lg = loop(fresh, 123, 12)
    assert more == ref_more and np.array_equal(lg, ref_lg)
    us2 = uniforms(12, 99)
    more, lg = eng.generate(more[-1], 12, pkg.engine.GEN_TYPICAL, temp, us2)
    ref_more, ref_lg = loop(fresh, ref_more[-1], 12, temp, us2)
    assert more == ref_more and np.array_equal(lg, ref_lg)
    assert_same_state(eng, fresh.state_download())
    eng.close()
    fresh.close()


@pytest.mark.parametrize("how", ["typical", "greedy"])
def test_stop_token_ends_the_run(pkg, make_model, how):
    eng = pkg.Engine(make_model(2, 768))
    temp, us = (2.0, uniforms(32, 21)) if how == "typical" else (None, None)
    ref_toks, _ = loop(eng, SEED_TOKEN, 32, temp, us)
    k = next((i for i in range(5, 32) if ref_toks[i] not in ref_toks[:i]), None)
    if k is None:
        pytest.skip("the reference run repeats every token it produces after step 5")
    eng.state_zero()
    loop(eng, SEED_TOKEN, k + 1, temp, us)
    ref_state = eng.state_download()
    eng.state_zero()
    mode = pkg.engine.GEN_TYPICAL if how == "typical" else pkg.engine.GEN_GREEDY
    toks, _ = eng.generate(SEED_TOKEN, 32, mode, temp or 1.0, us, stop=[ref_toks[k], 50276])
    assert toks == ref_toks[:k + 1]
    assert_same_state(eng, ref_state)
    eng.close()


@pytest.mark.parametrize("temp", [0.9, 0.3])
def test_kernel_token_equals_device_sampler(pkg, make_model, temp):
    eng = pkg.Engine(make_model(2, 768))
    us = uniforms(32, 8)
    tok, compared = SEED_TOKEN, 0
    for i in range(32):
        (got,), _ = eng.generate(tok, 1, pkg.engine.GEN_TYPICAL, temp, us[i:i + 1], want_logits=False)
        want, margin = eng.sample_typical(temp, float(us[i]))  # the same logits: those of the generate's forward
        if margin >= 1e-9:
            assert got == want, "step %d: generate %d, sample_typical %d" % (i, got, want)
            compared += 1
        tok = got
    assert compared >= 30
    eng.close()


def test_bad_arguments(pkg, make_model):
    eng = pkg.Engine(make_model(1, 768))
    T = pkg.engine.GEN_TYPICAL
    with pytest.raises(pkg.EngineError, match="out of range"):
        eng.generate(50277, 4, T, 0.9, uniforms(4, 1))
    with pytest.raises(pkg.EngineError, match="out of range"):
        eng.generate(1, 4, T, 0.9, uniforms(4, 1), stop=[7, 50277])
    with pytest.raises(pkg.EngineError, match="outside"):
        eng.generate(1, 4, T, 0.9, [0.5, 0.25, 1.0, 0.1])
    with pytest.raises(pkg.EngineError, match="n must be positive"):
        eng.generate(1, 0, T, 0.9, [])
    # nothing ran: the engine still decodes
    fresh = pkg.Engine(make_model(1, 768))
    assert eng.generate(1, 2, pkg.engine.GEN_GREEDY)[0] == loop(fresh, 1, 2)[0]
    fresh.close()
    eng.close()


def test_rwkv_generate_consumes_the_generator_like_the_sample_loop(pkg, make_model, tmp_path):
    """C++ surface: RWKV::generate(tok, n, temp) = the loop forward(tok); tok = sample(temp), including where the
    process-wide generator stands afterwards; also with a stop id that ends the run early."""
    exe = compile_cpp(os.path.join(ROOT, "tests", "helpers", "generate_gpu_test.cpp"), str(tmp_path / "generate_gpu_test"),
                      link_engine=True)
    r = subprocess.run([exe, make_model(2, 768)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ALL OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_pybind_generate_matches_forward_and_sample(pkg, make_model):
    import importlib
    import sys
    from util import PKG_DIR
    assert pkg.build.build_pybind()
    d = os.path.join(PKG_DIR, "bindings", "pybind")
    if d not in sys.path:
        sys.path.insert(0, d)
    os.environ["SO_LIB_PATH"] = "rwkv"
    binding = importlib.import_module("binding")
    model = binding.ModelWrapper(model_path=make_model(2, 768))
    ref, tok = [], SEED_TOKEN
    for _ in range(10):
        model.forward(tok)
        tok = int(model.get_output().argmax())
        ref.append(tok)
    model.init_state()
    assert model.generate(SEED_TOKEN, 10, greedy=True) == ref
    assert int(model.get_output().argmax()) == ref[-1]  # RWKV::out holds the last forward's logits
    model.init_state()
    toks = model.generate(SEED_TOKEN, 10, temp=0.9)
    assert len(toks) == 10 and all(0 <= t < 50277 for t in toks)
