"""CPU: the tiled-decode host logic (fastvideo_b200/vae_tiling.py) against outputs of the reference's own
ParallelTiledVAE.decode / tiled_decode / spatial_tiled_decode (oracle/gen_golden.py `tiling`, run around the cheap stand-in
decoder oracle/vae_ref.fake_tile_decode) -- bit-exact, fp32 and bf16 blends -- and the multi-rank tile distribution over
gloo against the serial result."""
import hashlib
import os
import socket
import sys

import pytest
import torch
import torch.multiprocessing as mp

from conftest import ROOT
from oracle.vae_ref import fake_tile_decode


def _sha(t):
    return hashlib.sha256(t.detach().float().cpu().contiguous().numpy().tobytes()).hexdigest()


def test_serial_tiling_matches_reference_bit_exactly(golden_dir):
    from fastvideo_b200 import vae_tiling
    g = torch.load(os.path.join(golden_dir, "vae_tiling.pt"))
    assert len(g["cases"]) >= 6
    for i, c in enumerate(g["cases"]):
        cfg = vae_tiling.TilingConfig(use_parallel_tiling=False, **c["cfg"])
        y = vae_tiling.decode(c["z"].clone(), fake_tile_decode, cfg)
        assert tuple(y.shape) == tuple(c["y_shape"]) and str(y.dtype) == c["y_dtype"], i
        assert _sha(y) == c["y_sha"], f"case {i}: tiled decode differs from the reference's"


def test_tile_plan_covers_every_tile_once():
    from fastvideo_b200 import vae_tiling
    cfg = vae_tiling.TilingConfig()
    for world in (1, 2, 3, 8):
        nt, nh, nw, ranges = vae_tiling.parallel_tile_plan((1, 16, 33, 135, 240), cfg, world)  # BASELINE config #5 latent
        assert (nt, nh, nw) == (11, 6, 10)
        seen = [g for a, b in ranges for g in range(a, b)]
        assert seen == list(range(nt * nh * nw))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    from fastvideo_b200 import vae_tiling
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(7)
        z = torch.randn(1, 12, 5, 40, 56)
        cfg = vae_tiling.TilingConfig()
        y = vae_tiling.decode(z, fake_tile_decode, cfg, rank=rank, world=world)
        # same tiles, same blend order, fp32 staging as in the reference's parallel path: equals the one-rank parallel path
        y1 = vae_tiling.parallel_tiled_decode(z, fake_tile_decode, cfg, 0, 1)[:, :, :17]
        # and for fp32 data the parallel result equals the serial temporal+spatial tiling
        ys = vae_tiling.decode(z, fake_tile_decode, vae_tiling.TilingConfig(use_parallel_tiling=False))
        bad = [f"{int((y != r).sum())} of {y.numel()} values differ from the {n} result"
               for n, r in (("one-rank parallel", y1), ("serial", ys)) if not torch.equal(y, r)]
        q.put((rank, "ok" if not bad and y.dtype == torch.float32 else f"MISMATCH ({y.dtype}): {bad}"))
    except Exception as e:  # noqa
        q.put((rank, f"FAIL {type(e).__name__}: {e}"))
    finally:
        dist.destroy_process_group()


def test_parallel_tiling_world2_gloo():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert all(r[1] == "ok" for r in res), res
