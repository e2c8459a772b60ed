#!/usr/bin/env python
"""bench.py -- tokens/s of single-batch decode through libcalm_b200.so (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one token of single-sequence decode (one pass of the per-token forward() path).  The
N = 1 workload is BASELINE.json configs[1]: Llama-3-8B shape, random-init fp8 (e5m2) weights, 4096-token
context, the timed tokens sitting at the END of the context (the reference's own "last tokens" protocol,
README.md:86) so attention reads the whole KV cache.  Every token streams all 7.5 GB of weights, far more
than the 126 MB L2, so no L2 flush is needed between steps.

Printed JSON (one line, rank 0):
  value      tokens/s with everything resident in HBM: device-side greedy loop (forward + argmax feeding
             the next token, no host round trip), CUDA events on the library's stream, max over ranks.
  e2e        tokens/s through the reference-facing C ABI with HOST buffers: forward_cuda(token, pos) per
             token, logits returned in host memory (device->host inside the timed region), greedy pick on
             the host, next token passed back in.  This is the call a calm user makes (run.c:209).
  roofline   dominant kernel: algorithmic bytes per launch / mean launch duration vs measured HBM peak.
  cpu_baseline  the reference's CPU implementation (oracle/_ref, or the oracle port) on this box's cores,
             bounded sample of the same workload.  Reported, not a target.
With --impl reference the same metric is measured on the reference's CPU path only (no product code).
For N > 1 the N GPUs serve ONE token stream, tensor-parallel (--parallel tp, the default): every rank holds 1/N of the
heads and FFN rows, the two partial projections per layer are summed inside k_matres over NVLink peer memory, the
classifier is split by vocabulary; "scaling": "strong".  --parallel replicas runs N independent copies instead
("scaling": "weak", no data-path collective).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi samples of SM clock / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8 or not (t0 <= ts <= t1 + 0.03):  # a line is printed up to one period after its sample
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


class RankAggregator:
    """Barrier / max-over-ranks / whole-job rate, the only cross-rank arithmetic of this bench (the replicas never
    exchange data on the hot path).  `dist` is torch.distributed (nccl on GPUs, gloo in the CPU test) or None."""

    def __init__(self, dist=None, device="cuda"):
        self.dist = dist
        self.device = device
        self.world = dist.get_world_size() if dist is not None else 1

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        if self.device != "cpu":
            import torch

            torch.cuda.synchronize()

    def max_over_ranks(self, v: float) -> float:
        if self.dist is None:
            return v
        import torch

        t = torch.tensor([v], device=self.device, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def whole_job_rate(self, steps: int, ms: float) -> float:
        """Units per second of the whole job: every rank processed `steps` units in at most `ms` milliseconds."""
        return self.world * steps / (ms / 1e3)


def dist_setup(n_gpus: int):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the path, nothing of ours on the path

def host_model(spec, seed):
    """The workload's model in host memory (generated on the GPU when there is one: 7.5 GB of randn is slow on CPU)."""
    import torch

    from calm_b200 import modelgen as mg

    dev = "cuda" if torch.cuda.is_available() else "cpu"
    t = mg.generate(spec, seed, device=dev)
    return mg.HostModel(spec, tensors=t, seq_len=4096 if spec.max_seq_len >= 4096 else None)


def numa_spread(model, threads):
    """Re-home the big weight tensors so that each OpenMP thread first-touches the rows it will later read (the
    reference's matmul splits rows statically over threads, infer.c:209-221): without this every page sits on the
    NUMA node of the thread that generated the model and a 2-socket host swings 9x between runs."""
    import ctypes as C

    import oracle
    import torch

    lib = C.CDLL(oracle._PATHS["port"])
    if not hasattr(lib, "oracle_parallel_copy"):
        return
    lib.oracle_parallel_copy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]
    for name, t in list(model.tensors.items()):
        if t.dim() < 2 or t.numel() * t.element_size() < (1 << 22):
            continue
        rows = int(np.prod(t.shape[:-1]))
        dst = torch.empty_like(t)  # untouched pages
        lib.oracle_parallel_copy(dst.data_ptr(), t.data_ptr(), rows, t.shape[-1] * t.element_size())
        model.tensors[name] = dst
    model.rebind()


def cpu_tokens_per_s(spec, seed, n_tokens, warmup, pos0, budget_s=None, model=None, threads=None):
    """Time the reference CPU forward() (oracle/_ref when it travelled, else the oracle port).
    Returns (tok/s, kind, threads, n_timed).  OMP_NUM_THREADS is ASSIGNED (torchrun exports 1 to its children)."""
    import oracle

    kind = "reference" if oracle.available("reference") else "port"
    if kind == "port" and not oracle.available("port"):
        oracle.build(ref=False)
    threads = threads or (os.cpu_count() or 1)
    os.environ["OMP_NUM_THREADS"] = str(threads)
    os.environ.setdefault("OMP_PROC_BIND", "true")
    model = model or host_model(spec, seed)
    if not getattr(model, "_spread", False):
        numa_spread(model, threads)
        model._spread = True
    ck = oracle.Checker(kind)
    ck.prepare(model)
    tok = 17
    for i in range(warmup):
        ck.forward(model, tok, pos0 + i)
    t0 = time.perf_counter()
    done = 0
    for i in range(n_tokens):
        logits = ck.forward(model, tok, pos0 + warmup + i)
        tok = int(np.argmax(logits))
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return done / dt, kind, threads, done


def run_reference_arm(args, spec):
    rank, world, local = dist_setup(args.gpus)
    if rank != 0:
        return
    pos0 = max(0, 4096 - args.steps - args.warmup)
    # every step is one token of the same workload; a wall-clock bound keeps a large --steps within minutes (the sample says how many ran)
    tps, kind, threads, done = cpu_tokens_per_s(spec, args.seed, args.steps, min(args.warmup, 4), pos0, budget_s=150.0)
    out = {
        "impl": "reference", "metric": "tok/s single-batch decode", "value": tps, "unit": "tok/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 / tps, "higher_is_better": True, "scaling": "strong" if (args.parallel == "tp" and args.gpus > 1) else "weak", "vs_baseline": None, "dtype": f"f32 ({spec.dtype} weights)",
        "data": "synthetic", "config": workload_config(spec, pos0, args),
        "cpu_baseline": {"value": tps, "unit": "tok/s", "cores": threads, "kind": kind,
                         "sample": f"{done} of {args.steps} steps (tokens) timed at pos {pos0 + min(args.warmup, 4)}.. of the same model, 150 s bound, all {threads} host threads"},
        "steps_timed": done,
        "e2e": {"value": tps, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def workload_config(spec, pos0, args):
    from calm_b200 import modelgen as mg

    per_gpu = mg.algorithmic_bytes(spec) / (args.gpus if (args.gpus > 1 and args.parallel == "tp") else 1)
    return {"workload": f"{spec.name}: {spec.n_layers} layers, dim {spec.dim}, hidden {spec.hidden_dim}, heads {spec.n_heads}/{spec.n_kv_heads}x{spec.head_dim}, "
                        f"vocab {spec.vocab_size}, {spec.dtype} weights, {'fp16' if getattr(args, 'kvbits', 16) == 16 else 'e5m2'} KV cache, context 4096, batch 1",
            "positions": f"{pos0}..{pos0 + args.steps + args.warmup - 1} (KV cache pre-filled to pos0)",
            "l2": f"inputs ({per_gpu / 1e9:.2f} GB of weights per step and GPU) exceed the 126 MB L2; no flush",
            "parallelism": "single GPU" if args.gpus <= 1 else (f"tp{args.gpus}" if args.parallel == "tp" else "replicas")}


# ------------------------------------------------------------------------------------------------

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="llama3-8b-fp8")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=20.0, help="seconds of CPU work for the cpu_baseline sample")
    ap.add_argument("--parallel", default="tp", choices=["replicas", "tp"],
                    help="N>1: ONE token stream tensor-parallel over the N GPUs (strong scaling; the two all-reduces per layer run "
                         "inside k_matres over NVLink peer memory; default) or independent replicas (weak scaling, no data-path collective)")
    ap.add_argument("--no-ref-cuda", action="store_true", help="skip timing the reference infer.cu (oracle/_ref/libcalm_ref_cuda.so) on this GPU")
    ap.add_argument("--kvbits", type=int, default=16, choices=[16, 8], help="KV cache element: fp16 (what the reference uses up to 4096 positions) or e5m2 (its choice beyond, run.c:537-539)")
    ap.add_argument("--layers", type=int, default=None, help="(debug) override the layer count")
    ap.add_argument("--pos0", type=int, default=None, help="(debug) first timed position instead of the end of the context")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write what they returned as DIR/<name>.npy: greedy_tokens (the device loop's tokens), "
                         "greedy_last_logits (its last step's logits), e2e_last_logits (forward_cuda's logits of the host-stepped loop's last step)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    from dataclasses import replace

    from calm_b200 import modelgen as mg

    spec = mg.SPECS[args.workload]
    if args.layers:
        spec = replace(spec, n_layers=args.layers)

    if args.impl == "reference":
        run_reference_arm(args, spec)
        return

    import torch

    from calm_b200 import lib

    rank, world, local = dist_setup(args.gpus)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    use_dist = world > 1
    dist = None
    if use_dist:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    agg = RankAggregator(dist if use_dist else None, device="cuda")
    barrier, max_over_ranks = agg.barrier, agg.max_over_ranks

    os.environ.setdefault("CALM_B200_QUIET", "1")  # keep stdout to the one JSON line
    sampler = ClockSampler(local)  # started well ahead of the timed region: nvidia-smi needs a second to come up on an 8-GPU box
    sampler.start()
    L = lib.load()  # built by build(): the bench compiles nothing, its tree may be read-only
    seq_len = 4096
    tp = None
    if use_dist and args.parallel == "tp":
        from calm_b200 import tp as ctp

        ctp.shard_dims(spec, world)  # raises when the shape does not split
        L.calm_b200_set_device(local)
        ident = [lib.tp_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        tp = (rank, world, ident[0])
    is_tp = tp is not None
    tensors = mg.generate(spec, args.seed + (0 if is_tp else rank), device="cuda")  # TP ranks hold the SAME model
    torch.cuda.synchronize()
    dm = lib.DeviceModel(spec, tensors, seq_len=seq_len, device=local, tp=tp, kvbits=args.kvbits)
    K, W = args.steps, args.warmup
    pos0 = max(0, seq_len - (K + W)) if args.pos0 is None else args.pos0
    dm.fill_kv(min(pos0, seq_len), seed=1 + rank)

    alg_bytes = mg.algorithmic_bytes(spec)
    kv_b = [mg.kv_bytes(spec, pos0 + W + i, seq_len, args.kvbits) for i in range(K)]
    bytes_per_tok = alg_bytes + float(np.mean(kv_b))

    # ---- leg 1: device-resident greedy decode (inputs resident in HBM)
    dm.decode_greedy(17, pos0, W)
    barrier()
    l0 = L.calm_b200_launch_count()
    t_wall0 = time.time()
    L.calm_b200_timer_start()
    toks = dm.decode_greedy(23, pos0 + W, K)
    ms = L.calm_b200_timer_stop()
    barrier()
    t_wall1 = time.time()
    launches = int(L.calm_b200_launch_count() - l0)
    dump = {"greedy_tokens": toks.astype(np.float64), "greedy_last_logits": dm.device_logits()} if args.dump_outputs else None
    ms = max_over_ranks(ms)
    value = K / (ms / 1e3) if is_tp else agg.whole_job_rate(K, ms)  # TP: the N GPUs serve ONE token stream

    # ---- leg 2: end to end through forward_cuda with host buffers
    tok = 23
    for i in range(W):
        p = dm.forward_raw(tok, pos0 + i)
        tok = int(np.argmax(np.ctypeslib.as_array(p, shape=(spec.vocab_size,))))
    barrier()
    t0 = time.perf_counter()
    tok = 23
    for i in range(K):
        p = dm.forward_raw(tok, pos0 + W + i)  # host int in -> host float[vocab] out
        tok = int(np.argmax(np.ctypeslib.as_array(p, shape=(spec.vocab_size,))))
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    if dump is not None and rank == 0:
        dump["e2e_last_logits"] = np.ctypeslib.as_array(p, shape=(spec.vocab_size,)).copy()
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    clocks = sampler.stop(t_wall0, time.time())  # both timed regions (device loop, then host-stepped loop)
    barrier()
    e2e = K / e2e_s if is_tp else agg.whole_job_rate(K, e2e_s * 1e3)

    # ---- roofline of the dominant kernel (per GPU: under tensor parallelism a rank streams 1/N of the layers and of the classifier)
    peak, peak_src = measured_peak()
    per_gpu = bytes_per_tok / (world if is_tp else 1)
    roof = dm_roofline(dm, L, spec, seq_len - 16, peak, peak_src, ms / K, per_gpu)

    out = {
        "metric": "tok/s single-batch decode", "value": value, "unit": "tok/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
        "higher_is_better": True, "scaling": "strong" if is_tp else "weak", "vs_baseline": None, "dtype": "f32 (fp8 e5m2 weights, f32 accumulate, fp16 KV)" if spec.dtype == "fp8" else f"f32 ({spec.dtype} weights)",
        "data": "synthetic", "config": workload_config(spec, pos0, args),
        "e2e": {"value": e2e, "unit": "tok/s", "h2d_bytes_per_step": 8, "d2h_bytes_per_step": spec.vocab_size * 4},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof,
        "algorithmic_gb_per_token": bytes_per_tok / 1e9, "algorithmic_gb_per_token_per_gpu": per_gpu / 1e9, "hbm_gbs_whole_token_per_gpu": per_gpu / 1e9 / (ms / K / 1e3),
        "frac_of_peak_whole_token": per_gpu / 1e9 / (ms / K / 1e3) / peak, "tp_mode": {0: None, 1: "ncclAllReduce between kernels", 2: "all-reduce inside k_matres over peer memory"}[L.calm_b200_tp_mode()],
    }
    if world == 1 and not spec.n_experts:
        # ---- the prompt pass (configs[2]: "2048-token prefill"): forward_prefill_cuda, tcgen05 GEMMs; timed with CUDA events on the library's stream
        try:
            n_pf = min(2048, seq_len)
            ptoks = np.array(mg.teacher_tokens(spec.vocab_size, n_pf), np.int32)
            served = dm.prefill(ptoks, 0)  # warm-up at the timed size: the pass's buffers are (re)allocated when a longer prompt arrives, tensor maps, attributes
            torch.cuda.synchronize()
            L.calm_b200_timer_start()
            dm.prefill(ptoks, 0)
            pf_ms = L.calm_b200_timer_stop()
            mm_params = spec.n_layers * ((spec.q_dim + 2 * spec.kv_dim) * spec.dim + spec.dim * spec.q_dim + 3 * spec.hidden_dim * spec.dim)
            flops = 2.0 * n_pf * mm_params + 2.0 * 2.0 * spec.n_layers * spec.q_dim * n_pf * (n_pf + 1) / 2
            tf = flops / (pf_ms / 1e3) / 1e12
            try:
                tpeak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"])
            except Exception:
                tpeak = 1400.0
            prefill = {"tokens": n_pf, "ms": pf_ms, "tok_s": n_pf / (pf_ms / 1e3), "tflops": tf, "frac_of_bf16_sustained": tf / tpeak,
                       "path": "tcgen05 GEMMs (f16 hi + lo activations: two MMAs per k-step) + block-causal attention" if served else "fed token by token (shape not served by the batched pass)",
                       "vs_serial_prompt": (n_pf / (pf_ms / 1e3)) / value}
        except Exception as e:
            prefill = {"unavailable": str(e)}
        out["prefill"] = prefill
    dm.close()

    if rank == 0 and world == 1 and not args.no_ref_cuda and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libcalm_ref_cuda.so")):
        # the kernel to beat (SURVEY.md s.6): the UNMODIFIED reference infer.cu on this GPU, same model, same positions, same
        # host-stepped protocol as the e2e leg; its own process (global statics, abort() on error), after ours released the device
        try:
            del tensors
            torch.cuda.empty_cache()
            r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ref_cuda_worker.py"), "--spec", args.workload, "--seq-len", str(seq_len), "--seed", str(args.seed),
                                "--bench", f"{pos0},{W},{K}"] + (["--layers", str(args.layers)] if args.layers else []), capture_output=True, text=True, timeout=600, cwd=ROOT)
            line = [l for l in r.stdout.splitlines() if l.startswith("{")]
            if r.returncode == 0 and line:
                rc = json.loads(line[-1])
                out["ref_cuda"] = {"e2e_tok_s": rc["tok_s"], "ms_per_step": rc["ms_per_step"], "ours_e2e_over_ref": e2e / rc["tok_s"],
                                   "what": "unmodified reference src/infer.cu (sm_100a build, oracle/_ref/libcalm_ref_cuda.so): forward_cuda per token, host argmax, same model and positions as e2e"}
            else:
                out["ref_cuda"] = {"unavailable": (r.stderr or r.stdout)[-300:]}
            tensors = None
        except Exception as e:
            out["ref_cuda"] = {"unavailable": str(e)}
            tensors = None

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            if tensors is None:
                tensors = mg.generate(spec, args.seed, device="cuda")
            hm = mg.HostModel(spec, tensors=tensors, seq_len=seq_len)
            del tensors
            ncpu = os.cpu_count() or 1
            tps, kind, threads, done = cpu_tokens_per_s(spec, args.seed, 10 ** 6, 1, seq_len - 64, budget_s=args.cpu_budget / 2, model=hm, threads=ncpu)
            tps2, _, threads2, done2 = cpu_tokens_per_s(spec, args.seed, 10 ** 6, 1, seq_len - 64, budget_s=args.cpu_budget / 2, model=hm, threads=max(1, ncpu // 2))
            if tps2 > tps:
                tps, threads, done, tps2, threads2, done2 = tps2, threads2, done2, tps, threads, done
            out["cpu_baseline"] = {"value": tps, "unit": "tok/s", "cores": threads, "kind": kind,
                                   "sample": f"{done} tokens at pos {seq_len - 63}.. of the same model ({args.cpu_budget / 2:.0f} s budget), {threads} threads, rows first-touched by "
                                             f"the thread that reads them; the other setting ({threads2} threads; reference default is nproc/2, infer.c:171-176): {tps2:.2f} tok/s"}
        except Exception as e:  # the baseline is reported, never required
            out["cpu_baseline"] = {"value": None, "unit": "tok/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
    if rank == 0:
        print(json.dumps(out), flush=True)
    if use_dist:
        dist.destroy_process_group()


def dm_roofline(dm, L, spec, pos, peak, peak_src, ms_per_tok, bytes_per_tok):
    """Roofline of the dominant kernel: the stage with the largest share of the token's time.  Launch durations come from
    %globaltimer stamps INSIDE the kernels of the production CUDA graph (first CTA past its dependency wait -> last CTA
    done; 8 extra tokens after the timed legs), so they describe the graph + PDL path that produced `value`."""
    stats, span_ms = dm.profile(23, pos, 8)
    total_ms = sum(v[0] for v in stats.values()) or 1.0
    table = {k: {"share": v[0] / total_ms, "us_per_launch": v[0] / max(v[2], 1) * 1e3, "gbs": (v[1] / 1e9 / (v[0] / 1e3)) if v[0] > 0 else None,
                 "frac": (v[1] / 1e9 / (v[0] / 1e3) / peak) if v[0] > 0 else None}
             for k, v in stats.items() if v[2] > 0}
    name, (ms, by, nl) = max(((k, v) for k, v in stats.items() if v[1] > 0), key=lambda kv: kv[1][0])
    achieved = by / 1e9 / (ms / 1e3) if ms > 0 else None
    # dram__bytes_read.sum + dram__bytes_write.sum per launch: not measurable in-run; the figure of the committed ncu capture is quoted with its source
    traffic, traffic_src = (117.53e6 + 3.41e6, "profiles/r02_ncu_full_one_layer.csv (k_ffn_up_ring<8,4,2>, Llama-3-8B fp8: dram__bytes_read.sum + dram__bytes_write.sum of one launch)") if (name == "matmul_ffn_up" and spec.name == "llama3-8b-fp8") else (None, None)
    return {"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if achieved else None,
            "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "bytes_per_launch": by / max(nl, 1), "us_per_launch": ms / max(nl, 1) * 1e3,
            "timing": "in-kernel %globaltimer stamps, production graph", "token_span_us_profiled": span_ms * 1e3, "stages": table}


if __name__ == "__main__":
    main()
