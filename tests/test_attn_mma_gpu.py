"""k_attn_mma (decode attention on mma.sync, head_dim 128 with 4 query heads per kv head) against the CPU oracle on
identical cache contents and against k_attn2 (CALM_B200_ATTN_MMA=0): the edges of the 16-position blocks, the slot
written during the token in the middle of a block, a backwards position step (the early copies were requested on a
stale kv_len), and the rolling cache with its re-rotated sinks, for the fp16 and the e5m2 cache."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from conftest import TOL_SIGMA  # noqa: E402
from test_scale_gpu import TOL8_SIGMA, fill_oracle_cache  # noqa: E402

from calm_b200 import lib  # noqa: E402
from calm_b200 import modelgen as mg  # noqa: E402

pytestmark = pytest.mark.gpu


def device_model(monkeypatch, mma, *args, **kw):
    """The switch is read when the model is prepared."""
    if mma:
        monkeypatch.delenv("CALM_B200_ATTN_MMA", raising=False)
    else:
        monkeypatch.setenv("CALM_B200_ATTN_MMA", "0")
    return lib.DeviceModel(*args, **kw)


def check(got, want, tol, what):
    sigma = float(want.std())
    err = float(np.abs(got - want).max())
    print(f"{what}: {err:.2e} = {err / sigma:.1e} sigma")
    assert err <= tol * sigma, (what, err, sigma)
    srt = np.sort(want)
    if srt[-1] - srt[-2] > 2 * tol * sigma:
        assert int(got.argmax()) == int(want.argmax()), what


@pytest.mark.parametrize("kvbits", [16, 8])
def test_block_edges_and_backwards_step(oracle_pkg, monkeypatch, kvbits):
    """Llama-3-8B's attention geometry (8 kv heads x 18 slices): kv_len 1, 16, 17, 18 and 4096 (block edges), kv_pos 2055
    (mid-block), then pos 4095 followed by pos 1000 in the same model (the early copies follow the previous kv_len)."""
    spec = mg.SPECS["attn-l8"]
    seq_len = 4096
    host = mg.HostModel(spec, seed=11, seq_len=seq_len, kvbits=kvbits)
    ck = oracle_pkg.Checker("port")
    tol = TOL_SIGMA if kvbits == 16 else TOL8_SIGMA
    steps = (0, 15, 16, 17, 2055, 4095, 1000)
    want = {}
    for pos in steps:
        ck.prepare(host)
        fill_oracle_cache(host, pos, seed=5, kvbits=kvbits)
        want[pos] = ck.forward(host, 17, pos)
        ck.release(host)
    got = {}
    for mma in (True, False):
        with device_model(monkeypatch, mma, spec, host.tensors, seq_len=seq_len, kvbits=kvbits) as dm:
            for pos in steps:
                dm.fill_kv(pos, seed=5)
                got[mma, pos] = dm.forward(17, pos)
    for pos in steps:
        check(got[True, pos], want[pos], tol, f"kv{kvbits} pos {pos} mma vs oracle")
        check(got[False, pos], want[pos], tol, f"kv{kvbits} pos {pos} k_attn2 vs oracle")
        check(got[True, pos], got[False, pos], tol, f"kv{kvbits} pos {pos} mma vs k_attn2")


@pytest.mark.parametrize("kvbits", [16, 8])
def test_rolling_cache_with_sinks(oracle_pkg, monkeypatch, kvbits):
    """A 16-position cache (one block) teacher-forced to pos 39: the ring slot and the 2 sinks are rewritten during
    the token and read from global memory over the early copy."""
    spec = mg.SPECS["tiny-llama"]
    toks = mg.teacher_tokens(spec.vocab_size, 40)
    host = mg.HostModel(spec, seed=1, seq_len=16, kvbits=kvbits)
    ref = oracle_pkg.teacher_forced(oracle_pkg.Checker("port"), host, toks)
    got = {}
    for mma in (True, False):
        with device_model(monkeypatch, mma, spec, host.tensors, seq_len=16, kvbits=kvbits) as dm:
            got[mma] = np.stack([dm.forward(t, i) for i, t in enumerate(toks)])
    # the sinks are re-rounded every step, which compounds (as in test_parity_gpu's rolling-cache test): 4x the tolerance
    tol = 4 * (TOL_SIGMA if kvbits == 16 else TOL8_SIGMA)
    sigma = float(ref.std())
    for mma in (True, False):
        err = float(np.abs(got[mma] - ref).max())
        print(f"kv{kvbits} rolling, {'mma' if mma else 'k_attn2'} vs oracle: {err / sigma:.1e} sigma")
        assert err <= tol * sigma
    err = float(np.abs(got[True] - got[False]).max())
    print(f"kv{kvbits} rolling, mma vs k_attn2: {err / sigma:.1e} sigma")
    assert err <= tol * sigma
