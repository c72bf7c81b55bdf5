"""bench.py's output contract (CPU part): `--impl reference` times the reference's CPU path (the staged unmodified reference, else the
oracle port) on a bounded sample and prints ONE JSON line with the keys the driver reads; under a multi-rank launch only rank 0 prints."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
            "data", "config", "cpu_baseline", "e2e", "gpu_launches"}


def run(extra_env=None):
    env = dict(os.environ, **(extra_env or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-sample", "8"],
                          capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_prints_one_contract_line():
    out = run()
    assert out.returncode == 0, out.stderr[-500:]
    lines = [l for l in out.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert REQUIRED <= set(d)
    assert d["impl"] == "reference" and d["unit"] == "labels/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "labels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_is_silent_on_other_ranks():
    out = run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_gpu_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


def test_dump_outputs_writes_float32_and_samples_large_outputs(tmp_path, monkeypatch):
    """bench.dump_outputs: one .npy per output, per-sequence arrays in float32 and scalars (the loss totals) in float64; above
    DUMP_BYTES the same seeded sequences of every per-sequence array, their indices, and the scalars whole."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    tok = torch.arange(40 * 15, dtype=torch.int64).view(40, 15)
    pad = tok % 3 == 0
    score = -torch.arange(40, dtype=torch.float32) / 7
    loss_sum, loss_basis = torch.tensor(123.456, dtype=torch.float32), torch.tensor(401, dtype=torch.int64)
    outputs = {"target": tok, "target_padding": pad, "target_score": score, "loss_sum": loss_sum, "loss_basis": loss_basis}
    bench.dump_outputs(str(tmp_path / "all"), outputs)
    got = {n: np.load(tmp_path / "all" / f"{n}.npy") for n in outputs}
    assert {n: a.dtype for n, a in got.items()} == {"target": np.float32, "target_padding": np.float32, "target_score": np.float32,
                                                    "loss_sum": np.float64, "loss_basis": np.float64}
    assert not (tmp_path / "all" / "rows.npy").exists()
    for n, t in outputs.items():
        assert np.array_equal(got[n], t.to(torch.float64).numpy()), n
    monkeypatch.setattr(bench, "DUMP_BYTES", 10 * (31 * 4 + 8) + 16)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outputs)
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.dtype == np.float64 and len(rows) == 10 and np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy"))
    r = rows.astype(np.int64)
    for n in ("target", "target_padding", "target_score"):
        assert np.array_equal(np.load(tmp_path / "a" / f"{n}.npy"), outputs[n].to(torch.float32).numpy()[r]), n
    for n in ("loss_sum", "loss_basis"):
        assert np.load(tmp_path / "a" / f"{n}.npy") == outputs[n].item(), n
    assert sum(os.path.getsize(tmp_path / "a" / f"{n}.npy") - 128 for n in (*outputs, "rows")) <= bench.DUMP_BYTES


def test_roofline_entry_reports_the_binding_roof():
    """bench.roof_entry: a GEMM class is measured against the roof that takes longer for its algorithmic work; an HBM class against
    the HBM roof; fractions are work / time / peak."""
    sys.path.insert(0, ROOT)
    import bench
    from novic_b200 import synth
    dims = synth.DecoderDims()
    peaks = {"hbm_gbs": 6500.0, "bf16_tflops_sustained": 1400.0}
    work = bench.algorithmic_work(4096, dims)
    gb = bench.gemm_hbm_bytes(4096, dims)
    rows, E, K, L = 4096 * (dims.prefix_len + dims.token_length - 2), dims.hidden_dim, dims.ffn_dim, dims.num_layers
    assert gb["fused_block"] == rows * L * 12 * E and gb["qkv_gemm"] == rows * L * 8 * E
    # the fused out-proj + feed-forward block: 0.78 MFLOP but 6 KB of rows per row and layer -> the HBM roof binds
    blk = bench.roof_entry("tensor", work["outproj_gemm"][1] + work["ffn1_gemm"][1] + work["ffn2_gemm"][1], gb["fused_block"], 2.0, 2.5, peaks)
    assert blk["bound"] == "hbm" and blk["unit"] == "GB/s" and blk["frac"] == blk["hbm_frac"] > blk["tensor_frac"]
    assert abs(blk["achieved"] - gb["fused_block"] / 2.0e-3 / 1e9) < 1e-6 and abs(blk["frac"] - blk["achieved"] / 6500.0) < 1e-12
    assert blk["isolated_frac"] < blk["frac"]
    # QKV and logits: the tensor roof binds
    for name in ("qkv_gemm", "logits_gemm"):
        e = bench.roof_entry("tensor", work[name][1], gb[name], 1.0, 1.2, peaks)
        assert e["bound"] == "tensor" and e["unit"] == "TFLOP/s" and e["frac"] == e["tensor_frac"] > e["hbm_frac"]
    a = bench.roof_entry("hbm", work["attention"][1], None, 2.0, 3.0, peaks)
    assert a["bound"] == "hbm" and "tensor_frac" not in a and abs(a["frac"] - work["attention"][1] / 2.0e-3 / 1e9 / 6500.0) < 1e-12
