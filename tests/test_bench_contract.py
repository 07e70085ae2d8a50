"""CPU: the bench.py contract on the one arm that runs without a GPU -- `--impl reference` (the reference's CPU block, or its
oracle port, timed on the host cores) must put exactly ONE JSON line on stdout with the keys the driver reads.
GPU (last test): the GPU arm's --steps and --dump-outputs on a one-layer model."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="8")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-sizes", "256,512"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "tokens/s"
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["vs_baseline"] is None and d["value"] > 0 and d["config"]["workload"]
    # "reference" when the reference's Python is importable (build container / staged copy), else the oracle port
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    ex = d["config"]["extrapolation"]
    assert ex["S"] == d["config"]["tokens"] == 75600 and ex["a"] > 0 and "S in" in d["cpu_baseline"]["sample"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_gpu_arm_refuses_to_run_without_cuda():
    """No CPU fallback on the product arm: without a CUDA device bench.py exits with an error and prints no result line."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("CUDA present")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert p.returncode != 0 and p.stdout.strip() == ""


def test_row_family_byte_models_accept_both_forward_call_shapes():
    """bench.py times the HBM-bound row / index kernels with algorithmic-byte work models; they are called with the argument
    lists of wan_dit.block_forward / vsa.video_sparse_attn_bshd (one GPU) and of distributed.py (sequence parallel: scatter
    variant with raw peer pointers, copy mode without weights, combine into out_segments)."""
    import torch
    import bench
    M, D, H, d, nblk = 128, 256, 2, 128, 2
    x = torch.zeros(M, D, dtype=torch.bfloat16)
    x32 = torch.zeros(M, D)
    qkv = torch.zeros(M, 4 * D, dtype=torch.bfloat16)
    assert bench.ln_bytes(x, None, None, eps=1e-6) == M * D * 4
    assert bench.ln_bytes(x32, None, None, x32[0], x32[0], eps=1e-6, want_hidden=True) == M * D * (4 + 2 + 2)
    assert bench.rope_bytes(qkv[:, :D], None, head_dim=d, eps=1e-6) == 2 * M * D * 2
    assert bench.rope_bytes(qkv[:, :D], None, qkv[:, D:2 * D], None, None, None, None, head_dim=d) == 4 * M * D * 2
    assert bench.rope_scatter_bytes(qkv[:, :D], None, qkv[:, D:2 * D], None, 1 << 40, 1 << 41, 8, None, None, None, None, head_dim=d) == 4 * M * D * 2
    assert bench.rope_scatter_bytes(qkv[:, :D], None, None, None, 1 << 40, 0, 8, None) == 2 * M * D * 2  # copy mode, one tensor
    q = torch.zeros(1, M, H, d, dtype=torch.bfloat16)
    assert bench.mean_bytes(q, nblk, None, None) == q.numel() * 2 + H * nblk * d * 2
    assert bench.mean_bytes(q, nblk, None, None, want_transposed=True) == q.numel() * 2 + 2 * H * nblk * d * 2
    sc = torch.zeros(H, nblk, nblk, dtype=torch.bfloat16)
    assert bench.softmax_bytes(sc) == 2 * sc.numel() * 2
    assert bench.topk_bytes(sc, 1, want_mask=False) == sc.numel() * (2 + 4)
    oc = torch.zeros(1, H, nblk, d, dtype=torch.bfloat16)
    assert bench.combine_bytes(q, oc, q, row_block=None, out=None, out_segments=(None, 64, (1, 2, 3))) == 3 * q.numel() * 2 + oc.numel() * 2
    assert bench.combine_bytes(q, oc, None) == 2 * q.numel() * 2 + oc.numel() * 2


def test_bad_step_counts_and_a_dump_from_the_cpu_arm_are_refused():
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "unused"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                           timeout=300, cwd=ROOT)
        assert p.returncode == 2 and p.stdout.strip() == "", (extra, p.stderr[-500:])


def test_dump_outputs_writes_float32_npy(tmp_path):
    import torch
    import bench
    x = torch.randn(2, 3, 5).bfloat16()
    bench.dump_outputs(str(tmp_path / "d"), {"noise_pred": x})
    y = np.load(tmp_path / "d" / "noise_pred.npy")
    assert y.dtype == np.float32 and np.array_equal(y, x.float().numpy())


@pytest.mark.gpu
def test_gpu_arm_steps_set_the_timed_steps_and_the_dump_is_reproducible(tmp_path):
    """Two runs with the same seeded inputs and different --steps: the timed region launches `steps` forwards (launch count
    scales exactly) and the two dumps agree as two bf16 roundings of the same values (separate processes are not
    guaranteed to be bit-equal)."""
    import torch
    from util import assert_two_bf16_paths_close
    lines, dumps = {}, {}
    for steps in (1, 2):
        d = tmp_path / f"steps{steps}"
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                            "--layers", "1", "--no-cpu-baseline", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-3000:]
        lines[steps] = json.loads(p.stdout.strip().splitlines()[-1])
        dumps[steps] = np.load(d / "noise_pred.npy")
    assert lines[1]["steps"] == 1 and lines[2]["steps"] == 2
    assert lines[1]["gpu_launches"] > 0 and lines[2]["gpu_launches"] == 2 * lines[1]["gpu_launches"]
    y = dumps[1]
    assert y.dtype == np.float32 and y.shape == (1, *lines[1]["config"]["latent"]) and np.isfinite(y).all()
    assert_two_bf16_paths_close(torch.from_numpy(dumps[2]), torch.from_numpy(y), name="noise_pred, --steps 2 vs 1")
