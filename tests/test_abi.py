"""CPU tests of the drop-in boundary: the C-ABI library loads, exports every symbol that
include/calm_b200.h declares, and the model records match the reference's layout.  No compute calls."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from conftest import ROOT  # noqa: E402

from calm_b200 import build as cbuild  # noqa: E402
from calm_b200 import cstructs, lib  # noqa: E402


@pytest.fixture(scope="module")
def L():
    cbuild.build()
    return lib.load()


def declared_functions():
    src = open(os.path.join(ROOT, "include", "calm_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"\b([a-z_0-9]+)\s*\([^;{]*\)\s*;", src)
    return [n for n in names if n not in ("defined",)]


def test_library_exports_every_declared_symbol(L):
    names = declared_functions()
    assert {"upload_cuda", "prepare_cuda", "forward_cuda", "perf_cuda"} <= set(names)
    for n in names:
        assert hasattr(L, n), f"libcalm_b200.so does not export {n}"
    assert set(names) == set(lib.SYMBOLS)
    assert L.calm_b200_abi_version() == 1


def test_no_oracle_in_product():
    """The product never routes through the checker: no source under calm_b200/ mentions oracle/, and the
    shared library has no dependency on it."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "calm_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".c", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text and "libcalm_oracle" not in text, f
    out = subprocess.run(["ldd", lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in out and "calm_ref" not in out


LAYOUT_PROG = r'''
#include <stdio.h>
#include <stddef.h>
#include HEADER
#define P(s, f) printf(#s "." #f " %zu\n", offsetof(struct s, f))
int main() {
  printf("Config %zu\nWeights %zu\nRunState %zu\nTransformer %zu\n", sizeof(struct Config), sizeof(struct Weights), sizeof(struct RunState), sizeof(struct Transformer));
  P(Config, dim); P(Config, hidden_dim); P(Config, head_dim); P(Config, n_layers); P(Config, n_heads); P(Config, n_kv_heads);
  P(Config, vocab_size); P(Config, seq_len); P(Config, rope_theta); P(Config, rotary_dim); P(Config, n_experts); P(Config, n_experts_ac);
  P(Config, norm_eps); P(Config, act_gelu); P(Config, norm_ln); P(Config, norm_par); P(Config, qkv_clip);
  P(Weights, dbits); P(Weights, token_embedding_table); P(Weights, rms_att_weight); P(Weights, rms_ffn_weight); P(Weights, wq); P(Weights, wk);
  P(Weights, wv); P(Weights, wo); P(Weights, w1); P(Weights, w2); P(Weights, w3); P(Weights, rms_final_weight); P(Weights, wcls); P(Weights, bqkv); P(Weights, moegate);
  P(RunState, x); P(RunState, he); P(RunState, att); P(RunState, exp); P(RunState, logits); P(RunState, kvbits); P(RunState, key_cache); P(RunState, value_cache);
  P(Transformer, config); P(Transformer, weights); P(Transformer, state); P(Transformer, n_params); P(Transformer, n_bytes); P(Transformer, n_bandwidth); P(Transformer, forward);
  printf("MAX_LAYERS %d MAX_EXPERTS %d KV_SINKS %d FF %d\n", MAX_LAYERS, MAX_EXPERTS, KV_SINKS, FF_UPDATE_KV_ONLY);
  return 0; }
'''


def struct_layout(header, workdir):
    """Sizes and field offsets of the model records declared by `header`, as printed by LAYOUT_PROG."""
    src = os.path.join(workdir, "l.c")
    with open(src, "w") as f:
        f.write(LAYOUT_PROG.replace("HEADER", '"%s"' % header))
    exe = os.path.join(workdir, "l")
    subprocess.run(["/usr/bin/gcc", src, "-o", exe], check=True)
    return subprocess.run([exe], capture_output=True, text=True, check=True).stdout


def test_struct_layout_matches_reference_header(tmp_path):
    """include/calm_model.h vs reference src/model.h, field by field (tests/golden/reference-layout.txt is the same
    program's output over the reference header, tools/make_golden.py); the ctypes mirror vs include/calm_model.h."""
    ours = struct_layout(os.path.join(ROOT, "include", "calm_model.h"), str(tmp_path))
    with open(os.path.join(ROOT, "tests", "golden", "reference-layout.txt")) as f:
        assert ours == f.read()
    kv = dict(line.rsplit(" ", 1) for line in ours.strip().splitlines()[:-1])
    for name, cls in (("Config", cstructs.Config), ("Weights", cstructs.Weights), ("RunState", cstructs.RunState), ("Transformer", cstructs.Transformer)):
        assert int(kv[name]) == C.sizeof(cls)
        for f, _ in cls._fields_:
            key = f"{name}.{f}"
            if key in kv:
                assert int(kv[key]) == getattr(cls, f).offset, key


def test_loading_fails_loudly_without_library(monkeypatch):
    monkeypatch.setattr(lib, "_lib", None)
    monkeypatch.setattr(lib, "LIB_PATH", "/nonexistent/libcalm_b200.so")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        lib.load()
