"""GPU: libfvb200's Video Sparse Attention against golden vectors produced by the REFERENCE'S OWN GPU KERNELS on a B200
(oracle/gen_golden_gpu.py: Triton fused_block_mean / fused_topk_mask / map_to_index / block-sparse forward, and the
reference's sm_100a kernel K1), committed as tests/golden/vsa_gpu_{small,720p,topk}.pt. Inputs are regenerated from the
recorded seeds. Tolerances are the reference's own gates (tests/test_block_sparse_sm100a.py:79-90: out max abs 0.02,
LSE max abs 0.05) plus this repo's bf16 rule for aggregate error (tests/util.py).

Also holds the oracle to the same fixtures on the CPU (-m "not gpu" part at the bottom of the file is in
tests/test_oracle_gpu_golden.py)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import vsa_index
from oracle.gen_golden_gpu import padded_inputs
from util import assert_two_bf16_paths_close, rel_l2

pytestmark = pytest.mark.gpu

OUT_ABS, LSE_ABS = 0.02, 0.05  # the reference's own gates for this kernel family


def _load(name):
    path = os.path.join(GOLDEN, name)
    if not os.path.exists(path):
        pytest.skip(f"{name} not generated yet (oracle/gen_golden_gpu.py)")
    return torch.load(path)


def _unpack_mask(packed, n):
    return torch.from_numpy(np.unpackbits(packed.numpy(), axis=-1)[..., :n].astype(bool))


@pytest.mark.parametrize("case", ["4x16x16_h2_randn", "5x6x7_h2_randn", "9x13x10_h2_randn"])
def test_small_grids_every_stage_against_the_reference_kernels(case):
    from fastvideo_b200 import ops, vsa
    fx = _load("vsa_gpu_small.pt")[case]
    q, k, v, gate, vbs, valid = padded_inputs(tuple(fx["shape"]), fx["heads"], fx["seed"], fx["flavour"])
    H, topk, nblk = fx["heads"], fx["topk"], vbs.numel()
    qd, kd, vd, gd, vbsd = (t.cuda() for t in (q, k, v, gate, vbs))
    vr = valid
    # (1) block means: same formula (fp32 sum / valid count -> bf16); summation order may differ in the last bit
    for n, x in (("q_c", qd), ("k_c", kd), ("v_c", vd)):
        mine = ops.block_mean(x.transpose(1, 2), nblk, None, vbsd).cpu()
        assert (mine != fx[n]).float().mean().item() < 5e-3, n
        assert rel_l2(mine, fx[n]) < 2e-3, n
    # (2) top-k map: bit-exact GIVEN THE REFERENCE'S SCORES (ties, bisection quirks and all)
    mine = ops.topk_mask(fx["scores"].cuda().contiguous(), topk).cpu()
    assert torch.equal(mine, fx["mask"])
    # (3) map -> index lists: bit-exact
    mi, mn = ops.map_to_index(fx["mask"].cuda())
    assert torch.equal(mi.cpu(), fx["q2k_idx"]) and torch.equal(mn.cpu(), fx["q2k_num"])
    # (4) sparse branch on the reference's lists vs the Triton kernel's output and LSE
    o, lse = ops.attention_blocklist(qd.transpose(1, 2), kd.transpose(1, 2), vd.transpose(1, 2), fx["q2k_idx"].cuda(),
                                     fx["q2k_num"].cuda(), kv_len=vbsd, q_len=vbsd, return_lse=True)
    o = o.transpose(1, 2).cpu()
    assert (o[:, :, vr].float() - fx["out_s"][:, :, vr].float()).abs().max().item() < OUT_ABS
    assert_two_bf16_paths_close(o[:, :, vr], fx["out_s"][:, :, vr], name="out_s vs Triton")
    fin = torch.isfinite(fx["lse"]) & vr[None, None]
    assert (lse.cpu()[fin] - fx["lse"][fin]).abs().max().item() < LSE_ABS
    assert (lse.cpu()[fin] - fx["lse"][fin]).abs().mean().item() < 1e-3
    if "k1_out" in fx:  # the reference's sm_100a kernel on the same lists
        assert (o[:, :, vr].float() - fx["k1_out"][:, :, vr].float()).abs().max().item() < OUT_ABS
    # (5) whole composite, reference signature
    out = vsa.video_sparse_attn(qd, kd, vd, vbsd, vbsd, topk, block_size=(4, 4, 4), compress_attn_weight=gd)
    _, aux = vsa.video_sparse_attn_bshd(qd.transpose(1, 2), kd.transpose(1, 2), vd.transpose(1, 2), vbsd, topk,
                                        gate=gd.transpose(1, 2), return_aux=True)
    same_rows = (aux["mask"].cpu().reshape(fx["mask"].shape) == fx["mask"]).all(-1)
    assert same_rows.float().mean().item() > 0.9
    rows = same_rows.repeat_interleave(64, 2) & vr[None, None]
    assert_two_bf16_paths_close(out.cpu()[rows], fx["out"][rows], name="video_sparse_attn")


@pytest.mark.parametrize("case", ["21x45x80_h2_local", "21x45x80_h2_randn"])
def test_720p_two_heads_topk144_against_the_reference_kernels(case):
    """BASELINE config #3's attention geometry (1440 tiles, 1100/320/20 of 64/16/4 tokens, top-k 144)."""
    from fastvideo_b200 import ops, vsa
    fx = _load("vsa_gpu_720p.pt")[case]
    q, k, v, gate, vbs, valid = padded_inputs(tuple(fx["shape"]), fx["heads"], fx["seed"], fx["flavour"])
    H, topk, nblk = fx["heads"], fx["topk"], vbs.numel()
    qd, kd, vd, gd, vbsd = (t.cuda() for t in (q, k, v, gate, vbs))
    blocks = fx["blocks"]
    rows = (blocks[:, None] * 64 + torch.arange(64)[None, :]).reshape(-1)
    vrows = valid[rows]
    mask = _unpack_mask(fx["mask_packed"], nblk)
    # block means over the whole tensor
    for n, x in (("k_c", kd),):
        mine = ops.block_mean(x.transpose(1, 2), nblk, None, vbsd).cpu()
        assert (mine != fx[n]).float().mean().item() < 5e-3, n
    # top-k on the reference's score rows
    mine = ops.topk_mask(fx["scores"].cuda().contiguous(), topk).cpu()
    assert torch.equal(mine, mask[:, :, blocks])
    # lists: ours from the reference's map == Triton's (count tensor stored in full, index tensor by hash)
    mi, mn = ops.map_to_index(mask.cuda())
    assert torch.equal(mn.cpu(), fx["q2k_num"])
    import hashlib
    assert hashlib.sha256(mi.cpu().contiguous().numpy().tobytes()).hexdigest() == fx["q2k_idx_sha"]
    # sparse branch at full size on the reference's lists; sampled q blocks compared
    o, lse = ops.attention_blocklist(qd.transpose(1, 2), kd.transpose(1, 2), vd.transpose(1, 2), mi, mn, kv_len=vbsd,
                                     q_len=vbsd, return_lse=True)
    o = o.transpose(1, 2).cpu()[:, :, rows]
    assert (o[:, :, vrows].float() - fx["out_s"][:, :, vrows].float()).abs().max().item() < OUT_ABS
    assert_two_bf16_paths_close(o[:, :, vrows], fx["out_s"][:, :, vrows], name="out_s vs Triton")
    l = lse.cpu()[:, :, rows]
    fin = torch.isfinite(fx["lse"]) & vrows[None, None]
    assert (l[fin] - fx["lse"][fin]).abs().max().item() < LSE_ABS
    if "k1_out" in fx:
        assert (o[:, :, vrows].float() - fx["k1_out"][:, :, vrows].float()).abs().max().item() < OUT_ABS
    # the composite: maps agree on most rows; outputs agree on rows whose lists agree
    out, aux = vsa.video_sparse_attn_bshd(qd.transpose(1, 2), kd.transpose(1, 2), vd.transpose(1, 2), vbsd, topk,
                                          gate=gd.transpose(1, 2), return_aux=True)
    my_mask = aux["mask"].cpu().reshape(mask.shape)
    same = (my_mask == mask).all(-1)
    assert same.float().mean().item() > 0.85, same.float().mean().item()
    sel = same[:, :, blocks].repeat_interleave(64, 2) & vrows[None, None]
    got = out.transpose(1, 2).cpu()[:, :, rows][sel]
    assert_two_bf16_paths_close(got, fx["out"][sel], name="video_sparse_attn 720p")


def test_topk_kernel_against_triton_on_tie_and_nonconvergence_stress_rows():
    from fastvideo_b200 import ops
    fx = _load("vsa_gpu_topk.pt")
    assert len(fx) >= 10
    for key, c in fx.items():
        mine = ops.topk_mask(c["scores"].cuda().contiguous(), c["topk"]).cpu()
        assert torch.equal(mine, c["mask"]), key


def test_k1_head_to_head_when_the_reference_kernel_is_present():
    """Side by side with the reference's sm_100a kernel K1: its output and LSE on the reference's own block lists, as
    oracle/gen_golden_gpu.py stored them in the fixtures (ragged and full grids, the 720p one on its sampled q blocks)."""
    from fastvideo_b200 import ops
    cases = [fx for name in ("vsa_gpu_small.pt", "vsa_gpu_720p.pt") for fx in _load(name).values() if "k1_out" in fx]
    assert len(cases) >= 4
    for fx in cases:
        q, k, v, _, vbs, valid = padded_inputs(tuple(fx["shape"]), fx["heads"], fx["seed"], fx["flavour"])
        nblk = vbs.numel()
        mask = fx["mask"] if "mask" in fx else _unpack_mask(fx["mask_packed"], nblk)
        blocks = fx.get("blocks", torch.arange(nblk))
        rows = (blocks[:, None] * 64 + torch.arange(64)[None, :]).reshape(-1)
        vr = valid[rows]
        vbsd = vbs.cuda()
        idx, num = ops.map_to_index(mask.cuda())
        o, lse = ops.attention_blocklist(*(t.cuda().transpose(1, 2) for t in (q, k, v)), idx, num, kv_len=vbsd, q_len=vbsd,
                                         return_lse=True)
        o = o.transpose(1, 2).cpu()[:, :, rows][:, :, vr]
        lse = lse.cpu()[:, :, rows][:, :, vr]
        assert (o.float() - fx["k1_out"][:, :, vr].float()).abs().max().item() < OUT_ABS, fx["shape"]
        assert (lse - fx["k1_lse"].reshape(lse.shape[:2] + vr.shape)[:, :, vr]).abs().max().item() < LSE_ABS, fx["shape"]
