"""CPU tests: the oracle (our restatement of reference infer.c) against the committed golden fixtures and the
stored outputs of reference runs (tools/make_golden.py); the synthetic-model writer against the reference loader."""
import hashlib
import json
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from conftest import KV_ATOL, KV_RTOL, ROOT, TOL_SIGMA, golden  # noqa: E402

from calm_b200 import modelgen as mg  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tools"))
from make_golden import GOLDEN_SPECS, load_ref_run, model_digest  # noqa: E402


@pytest.mark.parametrize("name", GOLDEN_SPECS)
def test_oracle_matches_golden(oracle_pkg, name):
    """Restatement vs fixtures produced by the unmodified reference (tools/make_golden.py)."""
    g = golden(name)
    spec = mg.SPECS[name]
    model = mg.HostModel(spec, seed=0)
    assert model_digest(model) == str(g["sha256"]), "synthetic model generator drifted from the one that made the fixtures"
    ck = oracle_pkg.Checker("port")
    logits = oracle_pkg.teacher_forced(ck, model, list(g["tokens"]))
    sigma = float(g["logits"].std())
    err = np.abs(logits[g["steps"]] - g["logits"]).max()
    assert err <= TOL_SIGMA * sigma, f"{name}: max |dlogit| {err:.3e} > {TOL_SIGMA * sigma:.3e}"
    safe = g["margin"] > 2 * TOL_SIGMA * sigma
    assert (logits.argmax(1)[safe] == g["argmax"][safe]).all()
    for l in range(spec.n_layers):
        for i, p in enumerate(g["kvpos"]):
            k, v = ck.read_kv(model, l, int(p))
            np.testing.assert_allclose(k, g["k"][l, i], rtol=KV_RTOL, atol=KV_ATOL)
            np.testing.assert_allclose(v, g["v"][l, i], rtol=KV_RTOL, atol=KV_ATOL)
    ck.release(model)


@pytest.mark.parametrize("name", ["tiny-fp8", "tiny-gf4", "tiny-qwen", "tiny-moe"])
def test_oracle_matches_reference_live(oracle_pkg, name):
    """Same comparison against a reference run on a different seed and at a position offset (golden reference-runs.npz:
    each step's largest logits and a fixed random sample of the others)."""
    spec = mg.SPECS[name]
    toks = mg.teacher_tokens(spec.vocab_size, 12, start=100)
    idx, ref, sigma = load_ref_run(name, 3, 12, start=100)
    for kind in ("port", "port_f64"):
        model = mg.HostModel(spec, seed=3)
        got = oracle_pkg.teacher_forced(oracle_pkg.Checker(kind), model, toks)
        assert np.abs(np.take_along_axis(got, idx, 1) - ref).max() <= TOL_SIGMA * sigma, kind


def test_oracle_rolling_cache(oracle_pkg):
    """Past seq_len the cache rolls with 2 pinned sinks (reference infer.c:330-332, 384-394)."""
    spec = mg.SPECS["tiny-fp8"]
    toks = mg.teacher_tokens(spec.vocab_size, 40)
    idx, ref, sigma = load_ref_run("tiny-fp8", 1, 40, seq_len=16)
    model = mg.HostModel(spec, seed=1, seq_len=16)
    got = oracle_pkg.teacher_forced(oracle_pkg.Checker("port"), model, toks)
    assert np.abs(np.take_along_axis(got, idx, 1) - ref).max() <= TOL_SIGMA * sigma


def test_decoders_exact(oracle_pkg):
    """fp8 = high byte of a half; gf4 = (q-4)*s/-4: numpy decoders, the oracle's C decoders and the
    quantiser must agree exactly (integer/bit work: bit-exact)."""
    import ctypes as C

    L = oracle_pkg.Checker("port").lib
    L.oracle_fp8_to_float.argtypes, L.oracle_fp8_to_float.restype = [C.c_uint8], C.c_float
    L.oracle_gf4_to_float.argtypes, L.oracle_gf4_to_float.restype = [C.c_uint32, C.c_int], C.c_float
    allb = np.arange(256, dtype=np.uint8)
    ref = mg.fp8_bytes_to_float(allb)
    got = np.array([L.oracle_fp8_to_float(int(b)) for b in allb], np.float32)
    finite = np.isfinite(ref)
    assert (ref[finite] == got[finite]).all()
    # torch's e5m2 agrees with the "high byte of half" reading for every finite value
    tv = torch.from_numpy(allb.copy()).view(torch.float8_e5m2).to(torch.float32).numpy()
    assert (tv[finite] == ref[finite]).all()
    rng = np.random.default_rng(0)
    words = rng.integers(0, 2 ** 32, size=512, dtype=np.uint64).astype(np.uint32)
    words = words[np.isfinite(mg.fp8_bytes_to_float((words & 0xFF).astype(np.uint8)))]
    dec = mg.gf4_words_to_float(words[None, :])[0].reshape(-1, 8)
    for i, w in enumerate(words[:64]):
        for k in range(8):
            assert dec[i, k] == np.float32(L.oracle_gf4_to_float(int(w), k))


def test_gf4_quantiser_properties():
    """Quantiser restated from convert.py:247-268: the scale element is reproduced exactly (code 0 ->
    (0-4)*s/-4 = s after e5m2 rounding) and every element is within 3/8 of the group scale (half a code
    step, plus the clamp of code 8 to 7 at the short positive end, plus the scale's own e5m2 rounding)."""
    g = torch.Generator().manual_seed(0)
    t = 0.02 * torch.randn(64, 256, generator=g)
    words = mg.to_gf4_words(t).numpy()
    dec = mg.gf4_words_to_float(words)
    tg = t.numpy().reshape(64, 32, 8)
    dg = dec.reshape(64, 32, 8)
    idx = np.abs(tg).argmax(-1)
    smax = np.take_along_axis(tg, idx[..., None], -1)[..., 0]
    s8 = torch.from_numpy(smax.copy()).to(torch.float8_e5m2).to(torch.float32).numpy()
    got = np.take_along_axis(dg, idx[..., None], -1)[..., 0]
    assert (got == s8).all()
    assert (np.abs(dg - tg) <= np.abs(s8)[..., None] * 0.375 + 1e-9).all()
    assert (mg.to_gf4_words(torch.zeros(2, 16)).numpy() != 0).sum() >= 0  # all-zero groups do not produce NaN
    assert np.isfinite(mg.gf4_words_to_float(mg.to_gf4_words(torch.zeros(2, 16)).numpy())).all()


def test_algorithmic_bytes_table():
    """n_bandwidth (run.c:523-532) of the five named shapes == BASELINE.md section 2."""
    exp = {"qwen2-0.5b-fp16": 0.988, "llama3-8b-fp8": 7.506, "llama3-8b-fp16": 15.010, "mistral-7b-gf4": 3.556,
           "mixtral-8x7b-fp8": 12.750, "llama3-70b-fp8": 69.507}
    for name, gb in exp.items():
        assert abs(mg.algorithmic_bytes(mg.SPECS[name]) / 1e9 - gb) < 2e-3, name
    assert abs(mg.kv_bytes(mg.SPECS["llama3-8b-fp8"], 4095, 4096) / 1e9 - 0.537) < 1e-3


def test_calm_file_loads_in_reference_driver(tmp_path, oracle_pkg):
    """A .calm file written by modelgen.write_calm is accepted by the UNMODIFIED reference program
    (tensors.c parser, run.c get_config/get_weights shape checks) and decodes on its CPU path: the file written now is
    byte for byte the one the reference program decoded (golden reference-run.json), and the oracle continues the
    prompt as the reference program did."""
    with open(os.path.join(ROOT, "tests", "golden", "reference-run.json")) as f:
        run = json.load(f)
    assert run["spec"] == "tiny-fp8" and run["seed"] == 0 and run["args"] == ["-n", "8", "-t", "0", "-i", "<|t7|><|t8|>"]
    spec = mg.SPECS["tiny-fp8"]
    model = mg.HostModel(spec, seed=0)
    path = str(tmp_path / "tiny.calm")
    mg.write_calm(path, spec, model.tensors)
    with open(path, "rb") as f:
        assert hashlib.sha256(f.read()).hexdigest() == run["calm_sha256"]
    # same greedy continuation from the oracle: prompt = BOS, 7, 8
    ck = oracle_pkg.Checker("port")
    m2 = mg.HostModel(spec, seed=0)
    ck.prepare(m2)
    toks = [spec.bos_id, 7, 8]
    for i, t in enumerate(toks):
        logits = ck.forward(m2, t, i)
    gen = []
    pos = len(toks)
    for _ in range(5):
        nxt = int(logits.argmax())
        gen.append(nxt)
        logits = ck.forward(m2, nxt, pos)
        pos += 1
    # the program prints the prompt after BOS, then the generated tokens
    assert run["tokens"][:2] == [7, 8] and run["tokens"][2:2 + len(gen)] == gen, (gen, run["tokens"])


def test_oracle_e5m2_cache_rounding_is_bit_exact(oracle_pkg):
    """oracle_round_e5m2 (the fp8 KV cache of reference infer.cu:476-481, __nv_fp8_e5m2(float): round to nearest even,
    saturate to the largest finite value) against torch's float8_e5m2 cast over normals, subnormals and ties."""
    import ctypes as C

    L = oracle_pkg.Checker("port").lib
    L.oracle_round_e5m2.argtypes, L.oracle_round_e5m2.restype = [C.c_float], C.c_float
    rng = np.random.default_rng(0)
    x = np.concatenate([rng.standard_normal(4000).astype(np.float32) * s for s in (1e-6, 1e-4, 1e-2, 1, 100, 1e4)] +
                       [np.array([0, -0.0, 57344, 57343.9, 2 ** -17, 2 ** -16 * 1.5, 2 ** -16 * 2.5, 1.25, 1.375, 1.5, -3.5], np.float32)])
    ref = torch.from_numpy(x).to(torch.float8_e5m2).to(torch.float32).numpy()
    got = np.array([L.oracle_round_e5m2(float(v)) for v in x], np.float32)
    assert np.array_equal(got, ref)
    assert L.oracle_round_e5m2(1e9) == 57344.0 and L.oracle_round_e5m2(-6e4) == -57344.0  # SATFINITE, where torch would give inf


def test_oracle_fp8_cache_mode_changes_only_the_cache(oracle_pkg):
    """kvbits == 8 in the oracle: same path, cache entries are e5m2 values; logits stay close to the fp16-cache run."""
    spec = mg.SPECS["tiny-fp8"]
    toks = mg.teacher_tokens(spec.vocab_size, 12)
    out = {}
    for kvbits in (16, 8):
        model = mg.HostModel(spec, seed=0, kvbits=kvbits)
        ck = oracle_pkg.Checker("port")
        out[kvbits] = oracle_pkg.teacher_forced(ck, model, toks)
        k, v = ck.read_kv(model, 1, 5)
        if kvbits == 8:
            for a in (k, v):
                assert np.array_equal(torch.from_numpy(a).to(torch.float8_e5m2).to(torch.float32).numpy(), a)
        ck.release(model)
    assert 0 < np.abs(out[8] - out[16]).max() < 0.5 * out[16].std()  # 2 mantissa bits per cache entry: visibly coarser, still the same function


def test_kv_fill_pattern_is_deterministic_and_bounded():
    a1, b1 = mg.kv_fill_pattern(3, 17, 32, seed=5)
    a2, b2 = mg.kv_fill_pattern(3, 17, 32, seed=5)
    assert np.array_equal(a1, a2) and np.array_equal(b1, b2) and a1.shape == (3, 17, 32)
    assert np.abs(a1).max() < 1 and np.abs(b1).max() < 1 and abs(float(a1.mean())) < 0.05 and not np.array_equal(a1, b1)
