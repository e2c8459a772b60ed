"""GPU parity at the scale of the headline configuration (VERDICT r01 #1): the full 4096-position context through the
multi-slice attention merge, the fp8 (e5m2) KV cache, and the 32-layer Llama-3-8B shape itself.

Checkers:
  * the CPU oracle (oracle/calm_oracle.c) given THE SAME cache contents: calm_b200_fill_kv's pseudo-random pattern is
    restated in numpy (modelgen.kv_fill_pattern) and written into the oracle's cache, so one oracle step at position p
    checks the device's attention over p cached positions without 4096 CPU steps;
  * the unmodified reference CUDA backend (oracle/_ref/libcalm_ref_cuda.so, tools/ref_cuda_worker.py), teacher-forced
    over the real context, for the full-size model and for kvbits == 8 (the reference CPU path has no fp8 cache); its
    logits are stored sampled under tests/golden/ (tools/make_golden.py --cuda).
Tolerances: fp16 cache: the stated 5e-3 sigma.  e5m2 cache: entries carry 2 mantissa bits, so a last-bit difference in
a k/v value before rounding moves a cache entry by up to 25 %; logits are compared at TOL8_SIGMA = 4e-2 sigma and the
cache entries themselves must be equal or adjacent e5m2 values."""
import ctypes as C
import os
import sys
from dataclasses import replace

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from conftest import ROOT, TOL_SIGMA, golden  # noqa: E402

from calm_b200 import lib  # noqa: E402
from calm_b200 import modelgen as mg  # noqa: E402
from calm_b200.cstructs import FF_UPDATE_KV_ONLY  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tools"))
from make_golden import ref_cuda_name  # noqa: E402

pytestmark = pytest.mark.gpu
TOL8_SIGMA = 4e-2


def fill_oracle_cache(model, n_pos, seed, kvbits):
    """Write calm_b200_fill_kv's pattern into the oracle's cache ([layer][pos][kv_dim] halves; e5m2 values when kvbits == 8)."""
    s = model.spec
    k, v = mg.kv_fill_pattern(s.n_layers * s.n_kv_heads, n_pos, s.head_dim, seed)

    def rnd(a):
        t = torch.from_numpy(a)
        return (t.to(torch.float8_e5m2).to(torch.float16) if kvbits == 8 else t.to(torch.float16)).numpy()

    st = model.transformer.state
    n = s.n_layers * model.seq_len * s.kv_dim
    for arr, ptr in ((k, st.key_cache), (v, st.value_cache)):
        dst = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint16)), shape=(n,)).view(np.float16).reshape(s.n_layers, model.seq_len, s.n_kv_heads, s.head_dim)
        src = rnd(arr).reshape(s.n_layers, s.n_kv_heads, n_pos, s.head_dim)
        dst[:, :n_pos] = src.transpose(0, 2, 1, 3)


@pytest.mark.parametrize("kvbits", [16, 8])
@pytest.mark.parametrize("spec_name", ["attn-l8", "tiny-hd256"])
def test_long_context_attention_vs_oracle(oracle_pkg, spec_name, kvbits):
    """Llama-3-8B's attention geometry (and a 256-wide multi-query head) at context positions up to 4095, device vs
    oracle on identical cache contents: the 18-slice merge, the transposing score path and the exponent accumulation
    over thousands of positions, compared value for value."""
    spec = mg.SPECS[spec_name]
    seq_len = 4096
    host = mg.HostModel(spec, seed=11, seq_len=seq_len, kvbits=kvbits)
    ck = oracle_pkg.Checker("port")
    tol = (TOL_SIGMA if kvbits == 16 else TOL8_SIGMA)
    with lib.DeviceModel(spec, host.tensors, seq_len=seq_len, kvbits=kvbits) as dm:
        for pos in (63, 1023, 2047, 4095):
            ck.prepare(host)
            fill_oracle_cache(host, pos, seed=5, kvbits=kvbits)
            want = ck.forward(host, 17, pos)
            ck.release(host)
            dm.fill_kv(pos, seed=5)
            got = dm.forward(17, pos)
            sigma = float(want.std())
            err = float(np.abs(got - want).max())
            print(f"{spec_name} kv{kvbits} pos {pos}: |cuda-oracle| {err:.2e} = {err / sigma:.1e} sigma")
            assert err <= tol * sigma, (pos, err, sigma)
            srt = np.sort(want)
            if srt[-1] - srt[-2] > 2 * tol * sigma:
                assert int(got.argmax()) == int(want.argmax())


@pytest.mark.parametrize("name", ["tiny-fp8", "tiny-llama", "tiny-gf4", "tiny-qwen", "tiny-moe"])
def test_fp8_kv_cache_teacher_forced_vs_oracle(oracle_pkg, name):
    """kvbits == 8 (what the unmodified reference driver selects for seq_len > 4096, run.c:537-539): teacher-forced
    logits vs the oracle's restatement of the e5m2 cache, the cache entries themselves, and the rolling cache."""
    spec = mg.SPECS[name]
    toks = mg.teacher_tokens(spec.vocab_size, 24)
    host = mg.HostModel(spec, seed=2, kvbits=8)
    ck = oracle_pkg.Checker("port")
    ref = oracle_pkg.teacher_forced(ck, host, toks)
    with lib.DeviceModel(spec, host.tensors, kvbits=8) as dm:
        got = np.stack([dm.forward(t, i) for i, t in enumerate(toks)])
        sigma = float(ref.std())
        err = float(np.abs(got - ref).max())
        print(f"{name} kv8: |cuda-oracle| {err:.2e} = {err / sigma:.1e} sigma")
        assert err <= TOL8_SIGMA * sigma
        for l in range(spec.n_layers):
            for p in (0, 5, 23):
                k, v = dm.read_kv(l, p)
                rk, rv = ck.read_kv(host, l, p)
                for a, b in ((k, rk), (v, rv)):  # equal or neighbouring e5m2 values (a rounding boundary can flip)
                    near = np.abs(a - b) <= 0.26 * np.maximum(np.abs(a), np.abs(b)) + 2e-5
                    assert near.all() and (a == b).mean() > 0.97
    ck.release(host)
    # rolling cache with re-rotated sinks on the fp8 cache
    toks = mg.teacher_tokens(spec.vocab_size, 40)
    host = mg.HostModel(spec, seed=1, seq_len=16, kvbits=8)
    ref = oracle_pkg.teacher_forced(ck, host, toks)
    with lib.DeviceModel(spec, host.tensors, seq_len=16, kvbits=8) as dm:
        got = np.stack([dm.forward(t, i) for i, t in enumerate(toks)])
    assert np.abs(got - ref).max() <= 4 * TOL8_SIGMA * ref.std()


@pytest.mark.parametrize("dtype", ["gf4", "fp8", "fp16"])
def test_ring_fed_kernels_vs_oracle(oracle_pkg, dtype):
    """Shapes the ring-fed stage kernels of ring.cuh serve (rows of whole 1 KB / 2 KB chunks, K-slices folded in shared memory;
    for gf4 with the staged group sums) against the CPU oracle, teacher-forced."""
    spec = replace(mg.SPECS["pf-tiny-hd128"], name="ring-" + dtype, dtype=dtype, dim=2048, hidden_dim=4096, n_heads=8, n_kv_heads=2, n_layers=2)
    toks = mg.teacher_tokens(spec.vocab_size, 20)
    host = mg.HostModel(spec, seed=7)
    ck = oracle_pkg.Checker("port")
    ref = oracle_pkg.teacher_forced(ck, host, toks)
    with lib.DeviceModel(spec, host.tensors) as dm:
        got = np.stack([dm.forward(t, i) for i, t in enumerate(toks)])
    ck.release(host)
    sigma = float(ref.std())
    err = float(np.abs(got - ref).max())
    print(f"ring-fed {dtype}: |cuda-oracle| {err:.2e} = {err / sigma:.1e} sigma")
    assert err <= TOL_SIGMA * sigma
    srt = np.sort(ref, 1)
    safe = (srt[:, -1] - srt[:, -2]) > 2 * TOL_SIGMA * sigma
    assert (got.argmax(1)[safe] == ref.argmax(1)[safe]).all()


def _ref_cuda(spec_name, layers, kvbits, seq_len, n, keep):
    """The reference CUDA backend's logits at `keep`, stored sampled (tools/make_golden.py --cuda): full-vocabulary std,
    argmax and top-2 margin, and the values at `idx` (its largest logits and a fixed random sample of the rest)."""
    g = golden(ref_cuda_name(spec_name, layers, kvbits, seq_len, n))
    assert list(g["keep"]) == keep
    return g


def _teacher_forced_device(spec, seed, n_tokens, keep, seq_len, kvbits):
    tensors = mg.generate(spec, seed, device="cuda")
    torch.cuda.synchronize()
    toks = mg.teacher_tokens(spec.vocab_size, n_tokens)
    out = {}
    with lib.DeviceModel(spec, tensors, seq_len=seq_len, kvbits=kvbits) as dm:
        for i, t in enumerate(toks):
            r = dm.forward(t, i, 0 if i in keep else FF_UPDATE_KV_ONLY)
            if i in keep:
                out[i] = r
    return np.stack([out[i] for i in keep])


def test_full_size_llama3_8b_at_bench_positions_vs_reference_cuda():
    """The headline workload itself: 32-layer Llama-3-8B shape, fp8 weights, fp16 cache, teacher-forced through the
    whole 4096-token context on both backends; logits at the bench's positions against the unmodified reference
    infer.cu on a B200."""
    keep = [63, 1023, 2047, 4071, 4095]
    ref = _ref_cuda("llama3-8b-fp8", None, 16, 4096, 4096, keep)
    got = _teacher_forced_device(mg.SPECS["llama3-8b-fp8"], 0, 4096, keep, 4096, 16)
    for i, p in enumerate(keep):
        sigma = float(ref["sigma"][i])
        err = float(np.abs(got[i][ref["idx"][i]] - ref["logits"][i]).max())
        print(f"llama3-8b-fp8 pos {p}: |ours - reference infer.cu| {err:.2e} = {err / sigma:.1e} sigma")
        # two GPU implementations, 32 layers of fp16-rounded cache entries between them: 2x the single-layer-stack tolerance
        assert err <= 2 * TOL_SIGMA * sigma
        if ref["margin"][i] > 4 * TOL_SIGMA * sigma:
            assert int(got[i].argmax()) == int(ref["argmax"][i])


@pytest.mark.parametrize("spec_name,layers,kvbits,seq_len,n", [("llama3-8b-fp8", 4, 8, 8192, 4200), ("mixtral-8x7b-fp8", 2, 16, 4096, 600), ("mistral-7b-gf4", 2, 8, 8192, 600)])
def test_reference_widths_vs_reference_cuda(spec_name, layers, kvbits, seq_len, n):
    """fp8 KV cache past 4096 positions (the reference driver's own switch), a Mixtral-width MoE and a Mistral-width
    gf4 model at reduced depth, against the unmodified reference CUDA backend."""
    keep = [0, n // 2, n - 1]
    ref = _ref_cuda(spec_name, layers, kvbits, seq_len, n, keep)
    spec = replace(mg.SPECS[spec_name], n_layers=layers)
    got = _teacher_forced_device(spec, 0, n, keep, seq_len, kvbits)
    tol = TOL_SIGMA if kvbits == 16 else TOL8_SIGMA
    for i, p in enumerate(keep):
        sigma = float(ref["sigma"][i])
        err = float(np.abs(got[i][ref["idx"][i]] - ref["logits"][i]).max())
        print(f"{spec_name}/{layers}L kv{kvbits} pos {p}: |ours - reference infer.cu| {err:.2e} = {err / sigma:.1e} sigma")
        assert err <= 2 * tol * sigma


def test_perf_cuda_reports_the_production_graph(capfd):
    """perf_cuda (reference infer.cu:761-801): per-stage time / GB/s from %globaltimer stamps inside the kernels of
    the SAME CUDA graph + PDL path that serves tokens; the stage sum must be consistent with the token span."""
    spec = replace(mg.SPECS["llama3-8b-fp8"], n_layers=4)
    tensors = mg.generate(spec, 0, device="cuda")
    with lib.DeviceModel(spec, tensors, seq_len=4096) as dm:
        dm.fill_kv(4000, seed=1)
        plain = [dm.forward_argmax(5, 4000 + i) for i in range(4)]
        stats, span_ms = dm.profile(5, 4000, 4)
        again = [dm.forward_argmax(5, 4000 + i) for i in range(4)]
        assert plain == again  # the stamped graph computes the same tokens
        total = sum(v[0] for v in stats.values()) / 4
        assert 0 < span_ms < 5 and 0.5 * span_ms <= total <= 1.6 * span_ms, (span_ms, total)
        for name in ("matmul_qkv", "attention", "matmul_attn", "matmul_ffn_up", "matmul_ffn_down", "output"):
            ms, by, nl = stats[name]
            assert nl == (4 if name == "output" else 16) and ms > 0 and by > 0
        L = lib.load()
        L.calm_b200_set_perf(1)
        dm.forward(5, 4000)
        L.perf_cuda()
        L.calm_b200_set_perf(0)
    out = capfd.readouterr().out
    assert "forward breakdown" in out and "matmul_ffn_up" in out and "GB/s" in out
