#!/usr/bin/env python
"""Generate tests/golden/*.npz by RUNNING THE REFERENCE (oracle/_ref/libcalm_ref_cpu.so, i.e. the
unmodified reference src/infer.c compiled with the reference's flags by oracle/Makefile).

The reference ships no golden vectors or unit tests (SURVEY.md s.4), so these fixtures are what pins
the oracle and the CUDA path on machines without /root/reference (the GPU box).  Each fixture holds,
for one seeded synthetic model (calm_b200.modelgen, seed 0) and the fixed teacher-forced token list:
  sha256     of the generated tensors (guards against a generator that drifted)
  tokens     the token list
  logits     float32 [n_keep, vocab] reference logits at the steps in `steps`
  argmax     int32 [n_tokens] reference greedy pick at every step
  margin     float32 [n_tokens] reference top-1 minus top-2
  k, v       float32 [n_layers, n_kvpos, kv_dim] KV-cache entries at positions `kvpos`

Besides the fixtures, what the tests compare with at other seeds and positions:
  reference-runs.npz       teacher-forced logits of the reference CPU backend per REF_RUNS case, sampled
  reference-run.json       the unmodified reference program decoding a .calm file written by modelgen.write_calm
  reference-layout.txt     sizes and offsets of the reference's model records (src/model.h; needs $REF = the
                           reference checkout, as in oracle/Makefile)
  ref-cuda-*.npz           (--cuda, on a B200) the reference CUDA backend at the widths of the real models, sampled

Run:  python tools/make_golden.py [--cuda] [name ...]     (name: a fixture or an output above without its extension)
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from calm_b200 import modelgen as mg  # noqa: E402

GOLDEN_SPECS = ["tiny-fp8", "tiny-fp16", "tiny-gf4", "tiny-qwen", "tiny-llama", "tiny-moe", "tiny-moe-gf4",
                "tiny-gelu-clip", "tiny-ln", "tiny-lnpar", "tiny-mha", "tiny-bias2", "tiny-hd256", "tiny-tp8", "tiny-tp8-moe", "ring-tp"]
N_TOKENS = 24
STEPS = [0, 1, 7, 15, 23]
KVPOS = [0, 5, 23]

# (spec, seed, n_tokens, first token index, seq_len): teacher_tokens(vocab, n_tokens, start) on HostModel(spec, seed, seq_len)
REF_RUNS = [(name, 3, 12, 100, None) for name in ("tiny-fp8", "tiny-gf4", "tiny-qwen", "tiny-moe")] + \
           [("tiny-fp8", 1, 40, 0, 16)] + \
           [(name, 5, 20, 50, None) for name in ("tiny-llama", "tiny-moe", "tiny-gf4")]
# logits kept per step of a REF_RUNS case (sampled(): keeps the fixtures small)
RUN_TOP, RUN_SAMPLE = 16, 48
# the .calm file the reference program decodes: spec, seed, program arguments after the file name
REF_PROGRAM = ("tiny-fp8", 0, ["-n", "8", "-t", "0", "-i", "<|t7|><|t8|>"])
# (spec, layers or None for all, kvbits, seq_len, n_tokens, kept positions): tools/ref_cuda_worker.py on the GPU
REF_CUDA_CASES = [("llama3-8b-fp8", None, 16, 4096, 4096, [63, 1023, 2047, 4071, 4095]),
                  ("llama3-8b-fp8", 4, 8, 8192, 4200, [0, 2100, 4199]),
                  ("mixtral-8x7b-fp8", 2, 16, 4096, 600, [0, 300, 599]),
                  ("mistral-7b-gf4", 2, 8, 8192, 600, [0, 300, 599])]
# logits kept per position of a ref-cuda case
CUDA_TOP, CUDA_SAMPLE = 64, 960


def model_digest(model) -> str:
    h = hashlib.sha256()
    for k in sorted(model.tensors):
        t = model.tensors[k]
        h.update(k.encode())
        h.update(t.contiguous().view(-1).view(__import__("torch").uint8).numpy().tobytes())
    return h.hexdigest()


def ref_run_key(name, seed, n_tokens, start=0, seq_len=None) -> str:
    return f"{name}:seed{seed}:start{start}:n{n_tokens}:seq{seq_len}"


def load_ref_run(name, seed, n_tokens, start=0, seq_len=None):
    """A stored REF_RUNS case: (idx, the reference's logits at idx [n_tokens, k], std of all its logits)."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "reference-runs.npz"))
    key = ref_run_key(name, seed, n_tokens, start, seq_len)
    return g[key + ".idx"], g[key + ".logits"], float(g[key + ".std"])


def sampled(logits, rng, top, n_random):
    """Per row of [rows, vocab] logits: the indices of its `top` largest entries and of `n_random` others drawn at random
    (sorted), and the logits there."""
    idx = []
    for row in logits:
        hi = np.argsort(row)[-top:]
        rest = np.setdiff1d(np.arange(len(row)), hi)
        idx.append(np.sort(np.concatenate([hi, rng.choice(rest, n_random, replace=False)])))
    idx = np.array(idx, np.int32)
    return idx, np.take_along_axis(logits, idx, 1).astype(np.float32)


def ref_cuda_name(spec, layers, kvbits, seq_len, n_tokens) -> str:
    return f"ref-cuda-{spec}-{layers or mg.SPECS[spec].n_layers}l-kv{kvbits}-ctx{seq_len}-n{n_tokens}"


def fixtures(only):
    ck = oracle.Checker("reference")
    outdir = os.path.join(ROOT, "tests", "golden")
    for name in GOLDEN_SPECS:
        if only and name not in only:
            continue
        spec = mg.SPECS[name]
        model = mg.HostModel(spec, seed=0)
        toks = mg.teacher_tokens(spec.vocab_size, N_TOKENS)
        logits = oracle.teacher_forced(ck, model, toks)
        srt = np.sort(logits, axis=1)
        k = np.zeros((spec.n_layers, len(KVPOS), spec.kv_dim), np.float32)
        v = np.zeros_like(k)
        for l in range(spec.n_layers):
            for i, p in enumerate(KVPOS):
                k[l, i], v[l, i] = ck.read_kv(model, l, p)
        np.savez_compressed(
            os.path.join(outdir, name + ".npz"), sha256=model_digest(model), tokens=np.array(toks, np.int32),
            steps=np.array(STEPS, np.int32), logits=logits[STEPS].astype(np.float32), argmax=logits.argmax(1).astype(np.int32),
            margin=(srt[:, -1] - srt[:, -2]).astype(np.float32), kvpos=np.array(KVPOS, np.int32), k=k, v=v)
        print(f"{name}: sigma {logits.std():.3f} min margin {(srt[:, -1] - srt[:, -2]).min():.2e}")


def reference_runs(path):
    out = {}
    rng = np.random.default_rng(0)
    for name, seed, n, start, seq_len in REF_RUNS:
        spec = mg.SPECS[name]
        model = mg.HostModel(spec, seed=seed, seq_len=seq_len)
        logits = oracle.teacher_forced(oracle.Checker("reference"), model, mg.teacher_tokens(spec.vocab_size, n, start))
        key = ref_run_key(name, seed, n, start, seq_len)
        out[key + ".idx"], out[key + ".logits"] = sampled(logits, rng, RUN_TOP, RUN_SAMPLE)
        out[key + ".std"] = np.float64(logits.std())
    np.savez_compressed(path, **out)


def reference_program(path):
    name, seed, args = REF_PROGRAM
    spec = mg.SPECS[name]
    with tempfile.TemporaryDirectory() as tmp:
        calm = os.path.join(tmp, "m.calm")
        mg.write_calm(calm, spec, mg.HostModel(spec, seed=seed).tensors)
        with open(calm, "rb") as f:
            digest = hashlib.sha256(f.read()).hexdigest()
        r = subprocess.run([os.path.join(ROOT, "oracle", "_ref", "run_ref"), calm] + args, capture_output=True, text=True, check=True,
                           env=dict(os.environ, CALM_CPU="1", OMP_NUM_THREADS="2"), timeout=120)
    tokens = [int(t) for t in r.stdout.splitlines()[-1].replace("<|t", " ").replace("|>", " ").split()]
    with open(path, "w") as f:
        json.dump({"spec": name, "seed": seed, "args": args, "calm_sha256": digest, "tokens": tokens}, f, indent=1)
        f.write("\n")


def reference_layout(path):
    ref = os.environ.get("REF")
    if not ref:
        print("reference-layout: set REF to the reference checkout")
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_abi import struct_layout

    with tempfile.TemporaryDirectory() as tmp:
        text = struct_layout(os.path.join(ref, "src", "model.h"), tmp)
    with open(path, "w") as f:
        f.write(text)


def ref_cuda(path, spec, layers, kvbits, seq_len, n, keep):
    """Logits of the reference CUDA backend at `keep`: full-vocabulary std, argmax and top-2 margin, and sampled() values."""
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "ref.npz")
        subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ref_cuda_worker.py"), "--out", out, "--spec", spec, "--seq-len", str(seq_len),
                        "--kvbits", str(kvbits), "--tokens", str(n), "--keep", ",".join(map(str, keep))] + (["--layers", str(layers)] if layers else []),
                       check=True, cwd=ROOT, timeout=900)
        logits = np.load(out)["logits"]
    idx, vals = sampled(logits, np.random.default_rng(0), CUDA_TOP, CUDA_SAMPLE)
    srt = np.sort(logits, axis=1)
    np.savez_compressed(path, keep=np.array(keep, np.int32), idx=idx, logits=vals, sigma=logits.std(1).astype(np.float64),
                        argmax=logits.argmax(1).astype(np.int32), margin=(srt[:, -1] - srt[:, -2]).astype(np.float32))


def main():
    args = sys.argv[1:]
    cuda = "--cuda" in args
    only = [a for a in args if a != "--cuda"]
    outdir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(outdir, exist_ok=True)
    if cuda:
        for spec, layers, kvbits, seq_len, n, keep in REF_CUDA_CASES:
            name = ref_cuda_name(spec, layers, kvbits, seq_len, n)
            if not only or name in only:
                ref_cuda(os.path.join(outdir, name + ".npz"), spec, layers, kvbits, seq_len, n, keep)
                print(name)
        return
    oracle.build(ref=True)
    fixtures(only)
    for name, make, ext in (("reference-runs", reference_runs, ".npz"), ("reference-run", reference_program, ".json"),
                            ("reference-layout", reference_layout, ".txt")):
        if not only or name in only:
            make(os.path.join(outdir, name + ext))
            print(name)


if __name__ == "__main__":
    main()
