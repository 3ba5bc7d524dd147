"""CPU: bench.py's host-side helpers — algorithmic FLOP formulas (BASELINE.md §3), synthetic batch layouts, the
thread calibration of the reference arm, and the JSON contract of `--impl reference` (no GPU involved)."""
import json
import os
import subprocess
import sys

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


@pytest.fixture()
def bench_mod(monkeypatch):
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self: self, raising=False)   # no CUDA in this container
    import bench
    return bench


def test_flops_per_pair_matches_baseline_md(bench_mod):
    T = bench_mod.PROMPT_LEN + bench_mod.RESP_LEN - 1 + 576
    assert T == 1135
    assert abs(bench_mod.flops_per_pair(T) / 1e12 - 92.45) < 0.05          # BASELINE.md §3: F_pair = 92.45 TFLOP


def test_synthetic_batches(bench_mod):
    b = bench_mod.synthetic_batch(0, 0, 2)
    ids, lab = b["concatenated_input_ids"], b["concatenated_labels"]
    assert ids.shape == (4, 560) and (ids == -200).sum(-1).tolist() == [1, 1, 1, 1] and int(ids[0, 35]) == -200
    assert (lab != -100).sum(-1).tolist() == [512] * 4 and torch.equal(ids[0, :48], ids[2, :48])   # pair shares prompt
    assert b["images"].shape == (2, 3, 336, 336)
    assert torch.equal(bench_mod.synthetic_batch(0, 0, 2)["concatenated_input_ids"], ids)            # seeded
    assert not torch.equal(bench_mod.synthetic_batch(1, 0, 2)["concatenated_input_ids"], ids)        # per-rank data
    from rlaifv_b200.omnilmm_model import omnilmm_dims
    d = omnilmm_dims()
    o = bench_mod.synthetic_omni_batch(0, 0, 2, d)
    oi = o["concatenated_input_ids"]
    assert oi.shape == (4, 625) and o["images"].shape == (2, 1024, 1792) and o["images"].dtype == torch.bfloat16
    assert int(oi[0, 35]) == d.im_start_token and int(oi[0, 36 + 64]) == d.im_end_token
    assert (oi == d.im_patch_token).sum(-1).tolist() == [64] * 4
    f = bench_mod.omni_flops_per_pair(d, 625)
    assert 50e12 < f < 60e12


def test_thread_calibration(bench_mod):
    n = bench_mod.usable_cores()
    assert 1 <= n <= (os.cpu_count() or 1)
    t = bench_mod.pick_cpu_threads()
    assert 1 <= t <= n and torch.get_num_threads() == t


def test_reference_arm_step_functions_run_at_tiny_dims(bench_mod):
    """Both step functions of the CPU arm (the staged unmodified reference, and the oracle-port fallback) complete an
    optimisation step; the reference one only where oracle/_ref has been staged (build() does it where the reference
    tree is readable)."""
    from oracle import llava_dpo_oracle as O
    from oracle import stage_ref
    makers = [bench_mod._port_step_fn]
    if stage_ref.available():
        makers.append(bench_mod._reference_step_fn)
    for make in makers:
        fn = make(2, cfg=O.TINY)
        l0, l1 = fn(), fn()
        assert l0 == l0 and l1 == l1 and l0 != l1            # finite, and the AdamW step changed the model
        ts = bench_mod._time_cpu_steps(fn, 1, 2)
        assert len(ts) == 2 and all(t > 0 for t in ts)


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun only rank 0 runs the CPU reference arm; the other ranks exit 0 without output."""
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_writes_seeded_float32_samples(bench_mod, tmp_path):
    """--dump-outputs: metrics plus parameter / gradient samples at the same seeded positions on every run, float32,
    within 64 MB for a full-size LLaVA-1.5-7B LoRA run (two stores of four arrays)."""
    import numpy as np
    from types import SimpleNamespace
    n = 3 * bench_mod.DUMP_SAMPLE

    def store(off):
        return SimpleNamespace(flat=torch.arange(n, dtype=torch.float32).to(torch.bfloat16),
                               grad=torch.full((n,), off, dtype=torch.bfloat16))
    policy = SimpleNamespace(store=store(1.0), lora=store(2.0))
    metrics = torch.arange(9, dtype=torch.float32)
    for d in ("a", "b"):
        bench_mod.dump_outputs(str(tmp_path / d), metrics, policy)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["grads.npy", "lora_grads.npy", "lora_params.npy", "metrics.npy", "params.npy"]
    for nm in names:
        a, b = np.load(tmp_path / "a" / nm), np.load(tmp_path / "b" / nm)
        assert a.dtype == np.float32 and np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / "a" / "metrics.npy"), metrics.numpy())
    assert np.load(tmp_path / "a" / "params.npy").shape == (bench_mod.DUMP_SAMPLE,)
    assert (np.load(tmp_path / "a" / "lora_grads.npy") == 2.0).all()
    assert sum(os.path.getsize(tmp_path / "a" / nm) for nm in names) <= 64 * 2 ** 20


def test_committed_bench_line_has_the_contract_keys():
    line = json.load(open(os.path.join(REPO, "profiles", "r01d_bench_n1.json")))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert k in line, k
    assert line["config"]["workload"].startswith("LLaVA-1.5-7B") and line["gpu_launches"] > 0
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(line["roofline"])
    assert {"value", "unit", "cores", "kind", "sample"} <= set(line["cpu_baseline"])
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
