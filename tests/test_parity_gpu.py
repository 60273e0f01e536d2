"""GPU parity: the CUDA engine (through the C ABI) vs the CPU oracle, and the oracle vs a stored run of the
unmodified reference CUDA build (tests/golden/reference/).

Tolerance (BASELINE.json north_star): logits within 1e-3 relative to the vector's
max-abs; argmax identical wherever the reference's own top-1/top-2 margin exceeds 1e-3
of max-abs (SURVEY.md H5: below that the reference's fp32 atomics decide the winner).
"""
import numpy as np
import pytest

from util import STATE_KEYS, load_reference, reference_logits_err, reference_margin, reference_state_err

pytestmark = pytest.mark.gpu

REL_TOL = 1e-3
SEED_TOKEN = 4118  # "###", first token of the storygen prompt


def make_engine(pkg, path, **kw):
    return pkg.Engine(path, **kw)


def rel_err(got, ref):
    return float(np.abs(got.astype(np.float64) - ref.astype(np.float64)).max() / max(np.abs(ref).max(), 1e-6))


def margin(ref):
    top = np.partition(ref, -2)[-2:]
    return float((top.max() - top.min()) / max(np.abs(ref).max(), 1e-6))


def run_pair(pkg, path, steps, threads=None):
    from oracle.oracle import Oracle
    eng = make_engine(pkg, path)
    orc = Oracle(path, threads=threads)
    tok, worst, checked_argmax = SEED_TOKEN, 0.0, 0
    for step in range(steps):
        got = eng.forward([tok])[0]
        ref = orc.forward(tok)
        e = rel_err(got, ref)
        worst = max(worst, e)
        assert e < REL_TOL, "step %d: logits rel err %.3g" % (step, e)
        if margin(ref) > 1e-3:
            assert int(got.argmax()) == int(ref.argmax()), "step %d argmax" % step
            checked_argmax += 1
        tok = int(ref.argmax())  # teacher forcing on the oracle's greedy stream
    st = eng.state_download()
    for k in ("xy", "aa", "bb", "dd"):
        ref = orc.state[k]
        scale = max(np.abs(ref).max(), 1e-6)
        assert np.abs(st[k] - ref).max() / scale < REL_TOL, "state %s" % k
    assert np.all(st["pp"] == 0.0)
    eng.close()
    orc.close()
    return worst, checked_argmax


@pytest.mark.parametrize("L,E,steps", [
    (2, 256, 6),     # CPL=2, half-empty lanes
    (3, 768, 8),     # 169M width: partial second chunk
    (2, 2048, 6),    # 1.5B width, CPL=4
    (2, 4096, 5),    # 7B width, CPL=8
    (1, 5120, 4),    # 14B width, CPL=10
])
def test_engine_matches_oracle(pkg, make_model, L, E, steps):
    worst, n = run_pair(pkg, make_model(L, E), steps)
    print("L=%d E=%d worst logits rel err %.3g (argmax checked on %d/%d steps)" % (L, E, worst, n, steps))


def test_169m_storygen_length(pkg, make_model):
    """BASELINE config: RWKV-4 169M shape (12 x 768), a longer decode."""
    worst, n = run_pair(pkg, make_model(12, 768), 24)
    print("169M worst rel err %.3g, argmax checked %d" % (worst, n))


def test_1b5_full_depth(pkg, make_model):
    """BASELINE config: RWKV-4 1.5B shape at full depth (24 x 2048)."""
    worst, n = run_pair(pkg, make_model(24, 2048), 6)
    print("1.5B worst rel err %.3g, argmax checked %d" % (worst, n))


def test_7b_full_size_bench_model(pkg):
    """The headline workload itself (32 x 4096, the file bench.py streams): three tokens against the oracle."""
    import sys
    from util import ROOT
    sys.path.insert(0, ROOT)
    import bench
    worst, n = run_pair(pkg, bench.model_path("7b", pkg), 3)
    print("7B worst rel err %.3g, argmax checked %d" % (worst, n))


def test_deterministic_across_runs(pkg, make_model):
    """Integer-limb accumulation has no reduction-order freedom: two runs are bit-identical."""
    path = make_model(2, 2048)
    outs = []
    for _ in range(2):
        e = pkg.Engine(path)
        toks, tok = [], SEED_TOKEN
        for _ in range(5):
            lg = e.forward([tok])[0]
            toks.append(lg.copy())
            tok = int(lg.argmax())
        outs.append(np.stack(toks))
        e.close()
    assert np.array_equal(outs[0], outs[1])


def test_forward_greedy_matches_host_argmax(pkg, make_model):
    path = make_model(2, 2048)
    e = make_engine(pkg, path)
    tok = SEED_TOKEN
    for _ in range(6):
        nxt, lg = e.forward_greedy(tok, want_logits=True)
        assert nxt == int(lg.argmax())
        tok = nxt
    e.close()


def test_decode_timed_streams(pkg, make_model):
    """The device-resident decode loops (bench.py `value`) compute the same tokens as forward()."""
    path = make_model(2, 2048)
    e = pkg.Engine(path)
    toks, tok = [], SEED_TOKEN
    for _ in range(6):
        toks.append(tok)
        tok = e.forward_greedy(tok)
    final = e.state_download()
    e.state_zero()
    assert e.decode_timed(toks, teacher_forced=True) > 0
    st = e.state_download()
    assert all(np.array_equal(st[k], final[k]) for k in st)
    e.state_zero()
    assert e.decode_timed([SEED_TOKEN] * 6, teacher_forced=False) > 0
    st = e.state_download()
    assert all(np.array_equal(st[k], final[k]) for k in st)
    e.close()


def test_state_roundtrip_and_restore(pkg, make_model):
    """Snapshot/restore through the host mirrors (RWKVState semantics, rwkv.h:173-240)."""
    path = make_model(2, 2048)
    e = pkg.Engine(path)
    for t in (SEED_TOKEN, 27, 1000):
        e.forward([t])
    snap = e.state_download()
    ref = e.forward([42])[0]
    e.forward([43])
    e.state_upload(snap)
    again = e.forward([42])[0]
    assert np.array_equal(ref, again)
    e.state_zero()
    z = e.state_download()
    assert all(np.all(z[k] == 0) for k in z)
    e.close()


def test_gpt_chunk_equals_token_by_token(pkg, make_model):
    """forward(vector, GPT) with maxGPT>1 returns per-token logits and the final state."""
    path = make_model(2, 2048)
    toks = [SEED_TOKEN, 5, 77, 31000]
    a = pkg.Engine(path, max_gpt=4)
    chunk = a.forward(toks, mode=1)
    sa = a.state_download()
    b = pkg.Engine(path)
    single = np.stack([b.forward([t])[0] for t in toks])
    sb = b.state_download()
    assert np.array_equal(chunk, single)
    n = a.n_layers * a.n_embed
    for k in ("xy", "aa", "bb", "dd"):
        assert np.array_equal(sa[k][:n], sb[k])
    a.close()
    b.close()


def test_parralel_mode_streams_are_independent(pkg, make_model):
    """MODE::PARRALEL: token t runs on state slot t (rwkv.cu:238-240)."""
    path = make_model(2, 2048)
    a = pkg.Engine(path, max_gpt=3)
    toks = [11, 222, 3333]
    first = a.forward(toks, mode=0)
    second = a.forward(toks, mode=0)
    b = pkg.Engine(path)
    for i, t in enumerate(toks):
        b.state_zero()
        assert np.array_equal(b.forward([t])[0], first[i])
        assert np.array_equal(b.forward([t])[0], second[i])
    a.close()
    b.close()


def test_errors(pkg, make_model, tmp_path):
    with pytest.raises(pkg.EngineError):
        pkg.Engine(str(tmp_path / "missing.bin"))
    bad = tmp_path / "short.bin"
    bad.write_bytes(np.array([2, 256], np.int64).tobytes() + b"\0" * 1000)
    with pytest.raises(pkg.EngineError):
        pkg.Engine(str(bad))
    e = pkg.Engine(make_model(2, 256))
    with pytest.raises(pkg.EngineError):
        e.forward([1, 2])  # chunk larger than max_gpt
    with pytest.raises(pkg.EngineError):
        e.forward([50277])  # token out of range
    e.close()


def test_oracle_vs_reference_cuda(pkg, make_model):
    """Pins the oracle: the UNMODIFIED reference (rwkv.cu + rwkv.h) run on a B200 on the same .bin and token
    stream, stored as tests/golden/reference/oracle_3x768.npz by tests/golden/make_reference_golden.py."""
    from oracle.oracle import Oracle
    ref = load_reference("oracle_3x768")
    assert ref["steps"].tolist() == list(range(8))
    toks = [int(t) for t in ref["tokens"]]
    path = make_model(3, 768)
    orc = Oracle(path)
    worst = 0.0
    for i, t in enumerate(toks):
        worst = max(worst, reference_logits_err(orc.forward(t), ref, i))
    print("oracle vs reference CUDA: worst logits rel err %.3g" % worst)
    assert worst < 1e-4
    for k in STATE_KEYS:
        assert reference_state_err(orc.state[k], ref, k) < 1e-4, k
    orc.close()
    # and the engine against the reference itself, same stream
    eng = pkg.Engine(path)
    for i, t in enumerate(toks):
        got = eng.forward([t])[0]
        assert reference_logits_err(got, ref, i) < REL_TOL
        if reference_margin(ref, i) > 1e-3:
            assert int(got.argmax()) == int(ref["argmax"][i])
    eng.close()


@pytest.mark.parametrize("L,E", [(2, 256), (3, 768), (2, 2048), (2, 4096), (1, 5120)])
def test_cluster_split_gather_is_bit_identical(pkg, make_model, L, E):
    """Thread-block clusters split the gather / quantisation and write each other's limb planes through
    distributed shared memory: the integers, hence the logits, must not change by a bit."""
    path = make_model(L, E)
    eng = make_engine(pkg, path)
    toks = [SEED_TOKEN, 17, 40000, 5, 291, 1023]

    def run():
        eng.state_zero()
        return np.stack([eng.forward([t])[0] for t in toks])

    base = run()
    tried = 0
    for c in (2, 4):
        try:
            eng.set_option("cluster", c)
        except pkg.EngineError as ex:  # the device cannot hold the grid in clusters of c
            print("cluster=%d not available: %s" % (c, ex))
            continue
        tried += 1
        got = run()
        assert np.array_equal(got, base), "cluster=%d changed the logits" % c
    eng.close()
    assert tried >= 1
