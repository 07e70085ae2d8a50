"""GPU, >= 2 devices: the DEFAULT multi-GPU path (push exchange: GEMM-epilogue / RoPE-pass / combine-kernel stores into
peer buffers at computed offsets, symmetric-memory barriers) and the NCCL fallback, against the single-rank engine, bit for
bit. Spawns torchrun on 2 (and 4, when present) ranks; skipped on a single-GPU machine. The workers report their verdicts
through a JSON file in the test's temporary directory."""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize("world", [2, 4])
def test_sp_forward_equals_single_rank_bit_for_bit(world, tmp_path):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, {torch.cuda.device_count()} visible")
    out = str(tmp_path / f"sp_parity_{world}.json")
    env = dict(os.environ, SP_WORKER_OUT=out)
    env.pop("FVB_SP_COMM", None)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "sp_worker.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert p.returncode == 0, (p.stdout[-3000:], p.stderr[-3000:])
    res = json.load(open(out))
    res_all = res
    sp = [r for r in res if not r.get("causal")]
    assert len(sp) == 8
    assert all(r["bit_equal_all_ranks"] for r in res if "skipped" not in r), res
    # the causal rollout on a head-sharded KV cache ran (keys are stored in a different order than on one rank, so it is
    # held to the bf16 parity rule against the reference's golden rollout instead of bit equality)
    assert any(r.get("causal") and "call" in r for r in res) or world > 2, res
    # the default request must really have run the push exchange (not silently fallen back)
    assert any(r["requested"] == "push" and r["used"] == "push" for r in res), res
