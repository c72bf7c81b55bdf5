#!/usr/bin/env python
"""Benchmark of the NOVIC decoder hot path: labels/sec, greedy decode, batch 4096 per GPU (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A step = one greedy decode (prefix prefill + 15 autoregressive steps, KV-cached) of one batch of 4096 synthetic
unit-norm 1024-d embeddings per GPU through novic_b200.PrefixedIterDecoder (random-init default decoder,
config/train.yaml:224-308).  Rank 0 prints ONE JSON line:
  value / e2e      weak scaling, 4096 embeddings per GPU (device-timed / through the public serving loop from pinned host memory)
  strong           (N > 1) the metric's own global batch of 4096 split N ways: 4096 / N embeddings per GPU
  secondary        BASELINE configs #3 (beam k = 3, 65 536 embeddings over 8 GPUs = 8192 per GPU), #4 (training step, global
                   batch 8192 over 8 GPUs = 1024 per GPU, embedding noise, NCCL gradient all-reduce, fused clip + AdamW) and #5
                   (CLIP ViT-H/14-378 image encoder + decoder, 1024 images per GPU) at this N
  roofline         per kernel class, against MEASURED_PEAKS.json, with ncu DRAM traffic from profiles/traffic.json
  cpu_baseline     (N = 1) the reference's own PrefixedIterDecoder.generate on the host cores over a bounded sample
`--impl reference` times the reference's CPU implementation alone: the unmodified reference staged in oracle/_ref (oracle/build_ref.py),
else the oracle port of its algorithm (re-forward schedule without KV cache).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH_PER_GPU = 4096
METRIC = "labels/sec (greedy, batch 4096)"
UNIT = "labels/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="K: timed steps of the headline greedy decode and of each of its three end-to-end "
                                                          "passes; the beam-search and training workloads time K clamped to 2..5 and 5..20 steps")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=("b200", "reference"))
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="embeddings per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=256, help="embeddings in the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary workloads (beam k=3, training step, image encoder + decoder)")
    ap.add_argument("--encoder-images", type=int, default=1024, help="images per GPU of the encoder + decoder workload (BASELINE config #5)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed greedy step returned (target ids, padding, scores; "
                                                          "with one GPU also loss_sum, loss_basis) as DIR/<name>.npy, to compare two builds "
                                                          "output for output; GPU arm only (not with --impl reference)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    return args


def workload_config(args, world):
    return {
        "workload": "BASELINE configs[1]: random-init default EmbeddingDecoder (E=512, FFN 128, L=6, 8 heads, P=4, V=6912, Cmax=16), "
                    f"{args.batch} synthetic unit-norm 1024-d embeddings per GPU, greedy decode (15 steps, tau=1, alpha=0), bf16 operands / fp32 accumulate",
        "batch_per_gpu": args.batch, "global_batch": args.batch * world, "gen_steps": 15, "parallelism": f"dp{world} (batch shards, final id gather)",
        "l2": "L2 flushed (256 MiB write) between timed iterations; per-step working set (KV cache 0.96 GB) also exceeds L2",
    }


# ----------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own greedy path on the host cores (staged copy oracle/_ref), else the oracle's restatement of it
# ----------------------------------------------------------------------------------------------------------------
def cpu_greedy_rate(sample: int, repeats: int = 1, warmup: int = 1):
    """Times `repeats` greedy decodes of `sample` embeddings on all host threads.  Returns (times [s], threads, kind, description).
    kind 'reference': embedding_decoder.PrefixedIterDecoder.generate of the unmodified reference, called exactly as infer.py:567-576
    does (collect_logits=False, calc_loss=True, tau=1, alpha=0); kind 'port': oracle.generate_greedy (same schedule: the whole
    sequence is re-forwarded every step, no KV cache)."""
    import contextlib
    from novic_b200 import synth
    torch.set_num_threads(os.cpu_count() or 1)
    dims = synth.DecoderDims()
    sd = synth.synth_state_dict(dims, seed=1)
    embed = synth.synth_embeddings(sample, seed=1234)
    os.environ["NOVIC_REFERENCE_ROOT"] = os.path.join(ROOT, "oracle", "_ref")     # never /root/reference at run time: it does not exist on the GPU box
    from oracle import refload
    kind = "port"
    fn = None
    if refload.available():
        try:
            with contextlib.redirect_stdout(sys.stderr):                            # the reference's logger writes to stdout; ours is one JSON line
                ref = refload.import_reference()
                model = refload.build_reference_decoder(ref, sd)
            fn = lambda e: model.generate(e, False, True, 1.0, 0.0, None, None, False)   # noqa: E731
            kind = "reference"
        except Exception as exc:                                                    # fall back to the port, say why
            print(f"bench.py: staged reference unusable ({type(exc).__name__}: {exc}); timing the oracle port", file=sys.stderr)
    if fn is None:
        from oracle import novic_oracle as orc
        cfg = orc.cfg_from_state_dict(sd)
        fn = lambda e: orc.generate_greedy(cfg, sd, e, 1.0, 0.0)                   # noqa: E731
    times = []
    with torch.inference_mode():
        for _ in range(warmup):
            fn(embed[: min(16, sample)])
        for _ in range(repeats):
            t0 = time.perf_counter()
            fn(embed)
            times.append(time.perf_counter() - t0)
    what = ("unmodified reference PrefixedIterDecoder.generate (oracle/_ref)" if kind == "reference" else "oracle port of the reference greedy path")
    desc = f"{what}, no KV cache, {sample} of the {BATCH_PER_GPU} embeddings per step (bounded sample), fp32, {torch.get_num_threads()} torch threads"
    return times, torch.get_num_threads(), kind, desc


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # the CPU arm runs on rank 0 only
    sample = args.cpu_sample
    times, cores, kind, desc = cpu_greedy_rate(sample, repeats=max(1, args.steps), warmup=max(1, min(args.warmup, 2)))
    ms = statistics.mean(times) * 1e3
    value = sample / (ms / 1e3)
    cfg = workload_config(args, max(1, args.gpus))
    cfg["workload"] = (f"BASELINE configs[1] on the host cores: random-init default EmbeddingDecoder (E=512, FFN 128, L=6, 8 heads, P=4, V=6912, Cmax=16), greedy decode "
                       f"(15 steps, tau=1, alpha=0) of a bounded sample of {sample} of the 4096 synthetic unit-norm 1024-d embeddings per step, fp32, the reference's "
                       "own schedule (whole sequence re-forwarded every step)")
    cfg.update(batch_per_gpu=None, global_batch=sample, parallelism=f"{cores} host threads", l2="n/a (CPU)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.rows.append(parts)

    def wait_started(self, timeout: float = 10.0) -> None:
        """nvidia-smi takes a while to attach; wait for its first sample so start-up does not perturb the timed region."""
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.05)

    def mark(self) -> None:
        self.rows.clear()   # keep only samples taken during the timed region

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------------
# algorithmic work per kernel class for one greedy decode of B embeddings (DESIGN.md section 5, SURVEY.md 8d)
# ----------------------------------------------------------------------------------------------------------------
def algorithmic_work(B: int, dims) -> dict:
    F, E, K, L, P, V, G = dims.embed_dim, dims.hidden_dim, dims.ffn_dim, dims.num_layers, dims.prefix_len, dims.vocab_size, dims.token_length - 1
    rows = B * (P + G - 1)                       # residual rows that pass through the layers (prefill P + G-1 decode steps)
    attn_bytes = 0
    attn_bytes += B * L * (P * 2 * E * 2 + 2 * P * E * 2)                    # prefill: K,V rows once + q in + out
    for s in range(P, P + G - 1):                                              # decode query at position s sees s+1 keys
        attn_bytes += B * L * ((s + 1) * 2 * E * 2 + 2 * E * 2)
    return {
        "embed_prep": ("hbm", B * F * (4 + 2)),
        "prefix_gemm": ("tensor", 2 * B * F * P * E),
        "qkv_gemm": ("tensor", 2 * rows * E * 3 * E * L),
        "attention": ("hbm", attn_bytes),
        "outproj_gemm": ("tensor", 2 * rows * E * E * L),
        "ffn1_gemm": ("tensor", 2 * rows * E * K * L),
        "ffn2_gemm": ("tensor", 2 * rows * K * E * L),
        "logits_gemm": ("tensor", 2 * B * G * E * V),
        "select": ("hbm", B * G * (-(-V // 64) * 32 + E * (4 + 4 + 2))),
    }


def gemm_hbm_bytes(B: int, dims) -> dict:
    """Algorithmic HBM bytes per decode of the GEMM classes: activation rows read and written once (bf16 operands 2 B, fp32 residual
    stream 4 B per element); weights (25 MB in all) stay L2-resident across the launches of a decode and are not counted.  A GEMM
    class is reported against whichever roof - tensor or HBM - takes longer for its algorithmic work (roof_entry)."""
    F, E, K, L, P, V, G = dims.embed_dim, dims.hidden_dim, dims.ffn_dim, dims.num_layers, dims.prefix_len, dims.vocab_size, dims.token_length - 1
    rows = B * (P + G - 1)
    return {
        "prefix_gemm": B * F * 2 + B * P * E * (4 + 2),                 # bf16 embedding in; fp32 residual rows + their LayerNorm-ed bf16 copy out
        "qkv_gemm": rows * L * (2 * E + 3 * 2 * E),                     # xn in; q, k, v out
        "outproj_gemm": rows * L * (2 * E + 4 * E + 4 * E + 2 * E),     # attention rows + residual in; residual + LN2 rows out
        "ffn1_gemm": rows * L * (2 * E + 2 * K),
        "ffn2_gemm": rows * L * (2 * K + 4 * E + 4 * E + 2 * E),
        "logits_gemm": B * G * (2 * E + -(-V // 64) * 32),              # final rows in; one 32-byte partial record per 64 vocabulary columns out
        # fused kernels keep their intermediates on chip: attention rows + residual in, residual + next LayerNorm rows out
        "fused_block": rows * L * (2 * E + 4 * E + 4 * E + 2 * E),
    }


def roof_entry(bound: str, amount: float, hbm_bytes, ms: float, iso_ms: float, peaks: dict) -> dict:
    """Roofline fields of one kernel class from its algorithmic work and its measured time per decode (ms in graph, iso_ms isolated).
    bound 'hbm': amount = bytes.  bound 'tensor': amount = FLOPs and, when hbm_bytes is given, the class is reported against the roof
    that takes longer for that work (the binding one); both fractions are kept as tensor_frac / hbm_frac."""
    def hbm(nbytes, t_ms):
        return nbytes / (t_ms * 1e-3) / 1e9
    def tensor(flops, t_ms):
        return flops / (t_ms * 1e-3) / 1e12
    if bound == "hbm":
        ach = hbm(amount, ms)
        return {"bound": "hbm", "achieved": ach, "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "isolated_frac": hbm(amount, iso_ms) / peaks["hbm_gbs"]}
    t_frac = tensor(amount, ms) / peaks["bf16_tflops_sustained"]
    out = {"bound": "tensor", "achieved": tensor(amount, ms), "unit": "TFLOP/s", "frac": t_frac,
           "isolated_frac": tensor(amount, iso_ms) / peaks["bf16_tflops_sustained"]}
    if hbm_bytes:
        h_frac = hbm(hbm_bytes, ms) / peaks["hbm_gbs"]
        out.update(tensor_frac=t_frac, hbm_frac=h_frac)
        if h_frac > t_frac:   # the HBM roof binds: moving the rows takes longer than the math
            out.update(bound="hbm", achieved=hbm(hbm_bytes, ms), unit="GB/s", frac=h_frac, isolated_frac=hbm(hbm_bytes, iso_ms) / peaks["hbm_gbs"])
    return out


def whole_decode_roofline(B: int, dims, ms_per_step: float, peaks: dict) -> dict:
    """The whole decode against both roofs (SURVEY.md 8d): algorithmic GEMM FLOPs vs the measured cuBLAS rate, algorithmic KV / row bytes of
    the attention vs the measured copy bandwidth, and the time the two would take back to back."""
    work = algorithmic_work(B, dims)
    flops = sum(v for k, (b, v) in work.items() if b == "tensor")
    nbytes = sum(v for k, (b, v) in work.items() if b == "hbm")
    t_tensor = flops / (peaks["bf16_tflops_sustained"] * 1e12) * 1e3
    t_hbm = nbytes / (peaks["hbm_gbs"] * 1e9) * 1e3
    return {"gemm_flops": flops, "hbm_bytes": nbytes, "tensor_ms": t_tensor, "hbm_ms": t_hbm, "frac_of_tensor_bound": t_tensor / ms_per_step,
            "frac_of_hbm_bound": t_hbm / ms_per_step, "frac_of_non_overlapped_bound": (t_tensor + t_hbm) / ms_per_step}


def _timed_decodes(model, embed, flush, n):
    """Mean device time (CUDA events on the launching stream, L2 flushed before each) of n greedy decodes."""
    total = 0.0
    for _ in range(n):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        model.generate(embed, False, True, 1.0, 0.0, None, None, False)
        b.record()
        torch.cuda.synchronize()
        total += a.elapsed_time(b)
    return total / n


def kernel_breakdown(model, embed, flush, steps: int, peaks: dict, dims) -> dict:
    """Two device timings of every kernel class, both with CUDA events on the launching stream:

    in_graph  - the captured decode graph with the launches of every OTHER class dropped (novic_debug_keep_classes), minus the same
                graph with no kernel at all: the class's launches run back to back with their real arguments, programmatic dependent
                launch and the L2 state of the decode, exactly as inside the product's graph.  This is `achieved` / `frac`.
    isolated  - direct launches (no graph) with an event pair around every launch: includes one launch gap per kernel (~2-3 us on a
                ~10 us kernel) - the pessimistic bound, comparable to ncu's serialised per-launch times in profiles/."""
    import ctypes as C
    from novic_b200 import _abi
    lib = _abi.lib()
    st = model._state(embed.device)
    names = list(_abi.KERNEL_CLASSES)
    with torch.inference_mode():
        # isolated: event pair per launch
        _abi.check(lib.novic_set_use_graphs(st["handle"], 0))
        model.generate(embed, False, True, 1.0, 0.0, None, None, False)
        torch.cuda.synchronize()
        _abi.check(lib.novic_kernel_timing(1))
        for _ in range(steps):
            model.generate(embed, False, True, 1.0, 0.0, None, None, False)
        n = len(names)
        ms = (C.c_double * n)()
        cnt = (C.c_int64 * n)()
        _abi.check(lib.novic_kernel_times(ms, cnt, n))
        _abi.check(lib.novic_kernel_timing(0))
        _abi.check(lib.novic_set_use_graphs(st["handle"], 1))
        # in graph: one class at a time
        in_graph = {}
        try:
            _abi.check(lib.novic_debug_keep_classes(st["handle"], 1 << 31))      # no kernel class at all: memsets, copies, host sync
            _timed_decodes(model, embed, flush, 2)
            base = _timed_decodes(model, embed, flush, steps)
            for i, name in enumerate(names):
                if cnt[i] == 0:
                    continue
                _abi.check(lib.novic_debug_keep_classes(st["handle"], 1 << i))
                _timed_decodes(model, embed, flush, 2)
                in_graph[name] = _timed_decodes(model, embed, flush, steps) - base
        finally:
            _abi.check(lib.novic_debug_keep_classes(st["handle"], 0))
        model.generate(embed, False, True, 1.0, 0.0, None, None, False)          # re-capture the full graph
    work = algorithmic_work(embed.shape[0], dims)
    if cnt[names.index('ffn1_gemm')] == 0:      # fused feed-forward kernel: its launches do both GEMMs of the block
        work["ffn2_gemm"] = ("tensor", work["ffn1_gemm"][1] + work["ffn2_gemm"][1])
    if cnt[names.index('outproj_gemm')] == 0:   # fused block kernel (out-proj + LN2 + feed-forward + LN): timed as class ffn2_gemm
        work["ffn2_gemm"] = ("tensor", work["ffn2_gemm"][1] + work["outproj_gemm"][1])
    gbytes = gemm_hbm_bytes(embed.shape[0], dims)
    if cnt[names.index('ffn1_gemm')] == 0 or cnt[names.index('outproj_gemm')] == 0:
        gbytes["ffn2_gemm"] = gbytes["fused_block"]
    total = sum(max(v, 0.0) for v in in_graph.values()) or 1.0
    out = {}
    for i, name in enumerate(names):
        if cnt[i] == 0:
            continue
        # classes of a few microseconds per decode drown in the run-to-run noise of the subtraction: never report less than
        # 40 % of the isolated time (the largest in-graph gain seen on any class is 45 %)
        iso_ms = ms[i] / steps
        g_ms = iso_ms if iso_ms < 0.1 else max(in_graph[name], 0.4 * iso_ms)   # (below 0.1 ms per decode the subtraction is all noise: keep the isolated time)
        entry = {"ms_per_step": g_ms, "launches_per_step": cnt[i] // steps, "share": g_ms / total, "isolated_ms_per_step": ms[i] / steps}
        if name in work:
            bound, amount = work[name]
            entry.update(roof_entry(bound, amount, gbytes.get(name), g_ms, iso_ms, peaks))
        out[name] = entry
    if cnt[names.index('outproj_gemm')] == 0 and 'ffn2_gemm' in out:
        # decode path with the fused block kernel (out-proj + LN2 + feed-forward + LN in one cluster kernel): name it for what it is
        out['block_outproj_ffn'] = out.pop('ffn2_gemm')
    return out


def load_peaks() -> dict:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "bf16_tflops": p["bf16_tflops"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops_sustained": 1400.0, "bf16_tflops": 1590.0, "source": "fallback (B200_PROFILING.md)"}


def traffic_entry(name: str):
    """ncu-measured DRAM traffic of one launch of a kernel class (profiles/traffic.json, written from `ncu --set full` captures by
    tools/ncu_traffic.py): {dram_bytes, algorithmic_bytes, ratio_to_algorithmic, tensor_pipe_pct, ...} or None."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.isfile(path):
        return None
    return json.load(open(path)).get(name)


DUMP_BYTES = 64 << 20


def dump_outputs(path: str, arrays: dict) -> None:
    """Writes each tensor as path/<name>.npy: per-sequence arrays (leading dimension = the first array's) in float32, where token ids
    below 2^24 and 0/1 padding flags are exact, and scalars in float64.  Outputs larger than DUMP_BYTES in all keep a fixed, seeded
    sample of the sequences, whose indices go to path/rows.npy."""
    import numpy as np
    arrays = {name: t.cpu().to(torch.float32 if t.ndim else torch.float64).numpy() for name, t in arrays.items()}
    n = next(iter(arrays.values())).shape[0]
    per_seq = [name for name, a in arrays.items() if a.ndim and a.shape[0] == n]
    row_bytes = sum(arrays[name].nbytes for name in per_seq) // n
    fixed_bytes = sum(a.nbytes for name, a in arrays.items() if name not in per_seq)
    if row_bytes * n + fixed_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, size=(DUMP_BYTES - fixed_bytes) // (row_bytes + 8), replace=False))
        arrays.update({name: arrays[name][rows] for name in per_seq})
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA (sm_100a) device: novic_b200 has no CPU fallback. Use --impl reference for the CPU arm.")
    # CPU leg first, on rank 0 of the single-GPU run only, before any other rank or collective exists (a rank spinning in a barrier
    # while rank 0 times the host cores would falsify it)
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        times, cores, kind, desc = cpu_greedy_rate(args.cpu_sample, repeats=1, warmup=1)
        cpu_baseline = {"value": args.cpu_sample / times[0], "unit": UNIT, "cores": cores, "kind": kind, "sample": desc + ", 1 run after warm-up"}
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from novic_b200 import EmbeddingNoise, _abi, default_decoder, synth
    from novic_b200.dist import gather_generation_async, gather_generation, train_step
    from novic_b200.optim import FusedAdamW
    from novic_b200.serve import GenerationPipeline
    dims = synth.DecoderDims()
    G = dims.token_length - 1
    model = default_decoder(dims, synth.synth_state_dict(dims, seed=1)).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lib = _abi.lib()

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(ms: float) -> float:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def greedy_workload(B: int):
        """(step_device, run_e2e, embed) for B embeddings per GPU."""
        embed_host = synth.synth_embeddings(B, seed=1234 + rank).pin_memory()
        embed = embed_host.to(dev)

        def step_device():
            if world == 1:
                tok, pad, _, loss_sum, loss_basis, score = model.generate(embed, False, True, 1.0, 0.0, None, None, False)
                return tok, pad, score, loss_sum, loss_basis
            # sharded: decode and gather are enqueued without a host synchronisation; the one sync of the step reads the global early-exit length
            tok, pad, score, T = model.generate_async(embed, 1.0, 0.0)
            tok, pad, score, T = gather_generation_async(tok.unsqueeze(1), pad.unsqueeze(1), score.unsqueeze(1), B * world, G, T)
            t = int(T.item())
            return tok[:, :, :t], pad[:, :, :t], score

        gather = (lambda t, p, sc, T: gather_generation_async(t, p, sc, B * world, G, T)) if world > 1 else None
        pipeline = GenerationPipeline(model, "greedy", post=gather, emit=(rank == 0))

        def run_e2e(steps):
            """The public serving loop (novic_b200.serve.GenerationPipeline): every step copies its batch from pinned host memory to the
            device, decodes it (and gathers across ranks), and rank 0 reads ids / padding / scores back to the host; the copies of
            neighbouring steps overlap the decode.  Timed as a whole: K steps between two synchronised CUDA events."""
            barrier()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = None
            for res in pipeline.run(embed_host for _ in range(steps)):
                out = res if res is not None else out
            b.record()
            torch.cuda.synchronize()
            barrier()
            return max_over_ranks(a.elapsed_time(b)), out
        return step_device, run_e2e, embed

    def timed(fn, steps):
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        barrier()
        torch.cuda.synchronize()
        n0 = lib.novic_launch_count()
        out = None
        for i in range(steps):
            flush.zero_()                      # L2 flush, outside the timed span
            starts[i].record()
            out = fn()
            ends[i].record()
        torch.cuda.synchronize()
        barrier()
        launches = lib.novic_launch_count() - n0
        per_step = [s.elapsed_time(e) for s, e in zip(starts, ends)]
        return max_over_ranks(sum(per_step)), launches, out, per_step

    W = max(args.warmup, 3)
    B = args.batch
    with torch.inference_mode():
        sampler = ClockSampler(local_rank) if rank == 0 else None
        step_device, run_e2e, embed = greedy_workload(B)
        for _ in range(W):
            step_device()
        run_e2e(W)
        if sampler:
            sampler.wait_started()
            sampler.mark()
        total_ms, launches, out, dev_steps = timed(step_device, args.steps)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, dict(zip(("target", "target_padding", "target_score", "loss_sum", "loss_basis"), out)))
        # three passes of exactly K steps each; the median pass is reported (all three are in e2e.runs_ms): one host hiccup in a 60 ms
        # loop (page-in after the previous process, a scheduler tick) otherwise decides the headline
        e2e_runs = [run_e2e(args.steps) for _ in range(3)]
        e2e_ms, out_host = sorted(e2e_runs, key=lambda r: r[0])[1]
        clocks = sampler.stop() if sampler else None
        tok = out[0]
        assert tok.shape[0] == B * world and tok.shape[-1] == G

        # ---- strong scaling on the metric's own batch: global 4096 embeddings, 4096 / N per GPU (SURVEY.md 8d)
        strong = None
        if world > 1 and B % world == 0:
            sd_step, sd_e2e, _ = greedy_workload(B // world)
            for _ in range(W):
                sd_step()
            sd_e2e(W)
            s_ms, _, s_out, _ = timed(sd_step, args.steps)
            s_e2e_ms = sorted(sd_e2e(args.steps)[0] for _ in range(3))[1]      # median of three K-step passes, like the headline figure
            assert s_out[0].shape[0] == B
            strong = {"scaling": "strong", "global_batch": B, "batch_per_gpu": B // world, "value": B * args.steps / (s_ms / 1e3), "unit": UNIT,
                      "ms_per_step": s_ms / args.steps, "e2e": {"value": B * args.steps / (s_e2e_ms / 1e3), "unit": UNIT, "ms_per_step": s_e2e_ms / args.steps}}

        # ---- BASELINE config #3: beam k = 3 over 65 536 embeddings sharded over 8 GPUs = 8192 per GPU (kept per GPU at every N)
        secondary = {}
        if not args.no_secondary:
            nb = 8192
            e_beam = synth.synth_embeddings(nb, seed=4321 + rank).to(dev)

            def beam_step():
                t, p, sc = model.generate_beam(e_beam, 3, 1.0, 0.0, None, False, 0.0, None, False)
                if world > 1:
                    t, p, sc = gather_generation(t, p, sc, nb * world, gen_len=G)
                return t
            beam_step()
            k_beam = max(2, min(args.steps, 5))
            b_ms, b_launches, b_out, _ = timed(beam_step, k_beam)
            assert b_out.shape[0] == nb * world and b_out.shape[1] == 3
            secondary["beam3"] = {"workload": f"BASELINE configs[2]: beam search k=3, tau=1, alpha=0, {nb} embeddings per GPU ({nb * world} in all; 65 536 at 8 GPUs), final gather of ids / padding / scores",
                                  "metric": "labels/sec (beam k=3)", "value": nb * world * k_beam / (b_ms / 1e3), "unit": UNIT, "ms_per_step": b_ms / k_beam, "steps": k_beam,
                                  "collective": "one all-gather of the packed results per step (none inside the decode loop)" if world > 1 else None}
            del e_beam

    # ---- BASELINE config #4: teacher-forced training step, 1024 samples per GPU (global 8192 at 8 GPUs), noise, all-reduce, clip + AdamW
    if not args.no_secondary:
        tb = 1024
        torch.manual_seed(1234)
        tmodel = default_decoder(dims, synth.synth_state_dict(dims, seed=1)).to(dev).train()        # input / layer dropout 0.1 (train.yaml defaults)
        opt = FusedAdamW(tmodel, lr=1.5e-3, betas=(0.9, 0.95), weight_decay=0.1)                     # train.yaml:427-441
        noise = EmbeddingNoise.create("GaussElemUniformAngle", 1024, 3.25, 45.0, 75.0, 0.0, 0.15)
        e_tr = synth.synth_embeddings(tb, seed=100 + rank).to(dev)
        tgt, pad = synth.synth_targets(tb, dims, seed=200 + rank)
        tgt, pad = tgt.to(dev), pad.to(dev)
        e_work = torch.empty_like(e_tr)

        def tr_step():
            e_work.copy_(e_tr)                 # the noise is applied in place (embedding_noise.py:50)
            return train_step(tmodel, opt, e_work, tgt, pad, None, noise=noise, gradient_clip=1.0)
        for _ in range(3):
            tr_step()
        k_tr = max(5, min(args.steps, 20))
        barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = lib.novic_launch_count()
        a.record()
        losses = [tr_step()[0] for _ in range(k_tr)]
        b.record()
        torch.cuda.synchronize()
        barrier()
        t_ms = max_over_ranks(a.elapsed_time(b))
        t_launches = lib.novic_launch_count() - n0
        coll_ms = None
        if world > 1:   # the gradient all-reduce on its own (50.9 MB fp32), for the record of what the overlap has to hide
            gb = tmodel._grad_bucket.flat
            for _ in range(2):
                dist.all_reduce(gb)
            torch.cuda.synchronize()
            a.record()
            for _ in range(5):
                dist.all_reduce(gb)
            b.record()
            torch.cuda.synchronize()
            coll_ms = max_over_ranks(a.elapsed_time(b)) / 5
        secondary["train_step"] = {
            "workload": f"BASELINE configs[3]: teacher-forced training step, {tb} samples per GPU ({tb * world} in all; 8192 at 8 GPUs), C=16 random targets, "
                        "GaussElemUniformAngle noise 3.25 / 45-75 deg / 0.15, dropout 0.1 / 0.1, forward + backward (CUDA graphs), NCCL all-reduce of the flat "
                        "gradient bucket in two parts (the first overlapping the backward pass), fused global-norm clip + AdamW, no host synchronisation",
            "metric": "training samples/sec", "value": tb * world * k_tr / (t_ms / 1e3), "unit": "samples/s", "ms_per_step": t_ms / k_tr, "steps": k_tr,
            "gpu_launches_per_step": t_launches / k_tr, "loss_first": losses[0].item(), "loss_last": losses[-1].item(),
            "collective": None if world == 1 else {"what": "ncclAllReduce of the 50.9 MB fp32 gradient bucket, timed alone", "ms": coll_ms},
        }
        del tmodel, opt

    # ---- BASELINE config #5: random-init CLIP ViT-H/14-378 image encoder + decoder end to end, 1024 synthetic 378 x 378 images per GPU
    if not args.no_secondary:
        from novic_b200.encoder import EncoderDecoder, ImageEncoder, VitDims, synth_images, synth_vit_state_dict
        vd = VitDims()
        enc = ImageEncoder(vd, images_per_chunk=64)
        enc.load_state_dict(synth_vit_state_dict(vd, seed=7))
        enc = enc.to(dev).eval()
        both = EncoderDecoder(enc, model)
        n_img = args.encoder_images
        base_img = synth_images(64, vd, seed=11 + rank).to(dev)
        images = base_img.repeat((n_img + 63) // 64, 1, 1, 1)[:n_img].contiguous()       # 64 distinct synthetic images, tiled to the batch
        Tk, Wd, Ly, Ml = vd.tokens, vd.width, vd.layers, vd.mlp_dim
        flops_img = 2 * Tk * Ly * (4 * Wd * Wd + 2 * Wd * Ml) + 4 * Tk * Tk * Wd * Ly + 2 * (Tk - 1) * 588 * Wd
        with torch.inference_mode():
            both.generate(images[:128])
            barrier()
            torch.cuda.synchronize()
            a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            n0 = lib.novic_launch_count()
            a.record()
            emb = both.embed(images)
            b.record()
            t5, p5, _, _, _, s5 = model.generate(emb, False, True, 1.0, 0.0, None, None, False)
            if world > 1:
                t5, p5, s5 = gather_generation(t5.unsqueeze(1), p5.unsqueeze(1), s5.unsqueeze(1), n_img * world, gen_len=G)
            c.record()
            torch.cuda.synchronize()
            barrier()
        e_ms, all_ms = max_over_ranks(a.elapsed_time(b)), max_over_ranks(a.elapsed_time(c))
        assert t5.shape[0] == n_img * world
        secondary["encoder_decoder"] = {
            "workload": f"BASELINE configs[4]: random-init CLIP ViT-H/14-378 image encoder (open_clip VisionTransformer as assumed in DESIGN.md: 730 tokens, width 1280, "
                        f"32 blocks, 16 heads x 80, MLP 5120, QuickGELU) + default decoder, {n_img} synthetic 378 x 378 images per GPU ({n_img * world} in all), images resident "
                        "in HBM, embeddings handed to the greedy decode on the device, final gather of ids",
            "metric": "images/sec (encode + greedy decode)", "value": n_img * world / (all_ms / 1e3), "unit": "images/s", "ms_per_step": all_ms, "steps": 1,
            "encoder_ms": e_ms, "encoder_tflops_per_gpu": flops_img * n_img / e_ms / 1e9, "encoder_frac_of_tensor_peak": flops_img * n_img / e_ms / 1e9 / load_peaks()["bf16_tflops_sustained"],
            "gflop_per_image": flops_img / 1e9, "gpu_launches": int(lib.novic_launch_count() - n0), "parity": "unpinned (un-vendored open_clip; oracle/vit_oracle.py restates the architecture)",
        }
        del enc, both, images, base_img

    if rank == 0:
        peaks = load_peaks()
        ms_per_step = total_ms / args.steps
        value = B * world * args.steps / (total_ms / 1e3)
        e2e_value = B * world * args.steps / (e2e_ms / 1e3)
        with torch.inference_mode():
            kernels = kernel_breakdown(model, embed, flush, min(args.steps, 5), peaks, dims)
        for name, entry in kernels.items():
            tr = traffic_entry(name)
            if tr:   # per-launch DRAM bytes from ncu beside the per-launch algorithmic bytes: traffic well below the algorithm's means L2 hits
                entry["traffic"] = {k: tr.get(k) for k in ("dram_bytes", "algorithmic_bytes", "ratio_to_algorithmic", "tensor_pipe_pct", "dram_pct", "capture")}
                if tr.get("ratio_to_algorithmic") is not None and tr["ratio_to_algorithmic"] < 0.6 and (tr.get("tensor_pipe_pct") or 0) < 30:
                    entry["regime"] = "latency-bound: neither DRAM traffic nor the tensor pipe is near its roof (dependent phases per tile)"
        dom = max(kernels, key=lambda k: kernels[k]["ms_per_step"])
        d = kernels[dom]
        tr = traffic_entry(dom)
        roofline = {"kernel": dom, "bound": d.get("bound"), "achieved": d.get("achieved"), "peak": peaks["hbm_gbs"] if d.get("bound") == "hbm" else peaks["bf16_tflops_sustained"],
                    "unit": d.get("unit"), "frac": d.get("frac"), "traffic": tr.get("dram_bytes") if tr else None, "regime": d.get("regime"), "peak_source": peaks["source"],
                    "how": "CUDA events on the launching stream around the captured decode graph with only this kernel class's launches kept (real arguments, PDL, L2 flushed "
                           "before each decode), minus the same graph with no kernels; achieved = algorithmic work of the class's launches / that duration, i.e. per-launch work / average "
                           "launch duration.  isolated_* = event pair around every direct launch (adds a launch gap per kernel; comparable to ncu's serialised times in profiles/).  "
                           "traffic = dram__bytes_read.sum + dram__bytes_write.sum of one launch from an ncu --set full capture (profiles/traffic.json)",
                    "whole_decode": whole_decode_roofline(B, dims, ms_per_step, peaks),
                    "kernels": kernels}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(args, world), "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms / args.steps, "runs_ms": [round(r[0], 3) for r in e2e_runs],
                    "h2d_bytes_per_step": B * dims.embed_dim * 4, "d2h_bytes_per_step": int(sum(t.numel() * t.element_size() for t in out_host)),
                    "api": "novic_b200.serve.GenerationPipeline.run (double-buffered H2D / D2H around PrefixedIterDecoder.generate; per-rank H2D, rank 0 reads the gathered result)"},
            "gpu_launches": int(launches), "roofline": roofline,
            "step_ms": {"device_median": statistics.median(dev_steps), "device_max": max(dev_steps), "device_min": min(dev_steps)},
        }
        if strong is not None:
            line["strong"] = strong
        if secondary:
            line["secondary"] = secondary
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
