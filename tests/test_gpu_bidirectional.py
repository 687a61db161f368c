"""F5: bidirectional flow with forward-backward occlusion masks (RAFT.forward_backward, rb_flow_consistency).

The two directions run as one batch of 2B pairs, and a batch never mixes samples (DESIGN.md section 4), so each half of
the result must equal a plain forward call bit for bit; the masks are checked against the kernel called through the
ABI on the returned flows, and the kernel against the fp64 oracle."""
import importlib.util
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))  # fb_oracle.py sits beside the tests
from fb_oracle import fb_consistency  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _model(cuda, small, H, W, iters, B=1, volume_free=None):
    from raft_b200 import synth
    from networks.RAFT import RAFT
    return RAFT((H, W, 3), SimpleNamespace(small=small), iters=iters, batch=B, device=cuda,
                volume_free=volume_free).load(synth.make_weights(small))


def _abi_consistency(flow_fw, flow_bw, scale, alpha1=0.01, alpha2=0.5):
    from raft_b200 import capi
    B, H, W, _ = flow_fw.shape
    fw, bw = flow_fw.contiguous(), flow_bw.contiguous()
    occ_fw = torch.full((B, H, W), 255, dtype=torch.uint8, device=fw.device)
    occ_bw = torch.full_like(occ_fw, 255)
    with torch.cuda.device(fw.device):
        capi.check(capi.lib.rb_flow_consistency(capi.ptr(fw), capi.ptr(bw), capi.ptr(occ_fw), capi.ptr(occ_bw), B, H, W,
                                                scale, alpha1, alpha2, capi.stream()))
    torch.cuda.synchronize()
    return occ_fw, occ_bw


@pytest.mark.parametrize("small,B,H,W,u8,use_graph,volume_free", [
    (False, 1, 64, 96, False, True, False),
    (True, 1, 64, 96, False, True, False),
    (False, 2, 60, 100, True, True, False),
    (True, 2, 60, 100, False, False, False),
    (False, 1, 60, 100, False, False, False),
    (False, 2, 64, 96, False, True, True),
    (True, 1, 60, 100, True, True, True),
])
def test_halves_equal_forward_calls_bit_exact(cuda, small, B, H, W, u8, use_graph, volume_free):
    from raft_b200 import synth
    iters = 3
    l, r = synth.make_batch(B, H, W)
    if u8:
        l, r = (np.round(x * 255).astype(np.uint8) for x in (l, r))
    bi = _model(cuda, small, H, W, iters, B, volume_free)
    bi.engine().use_graph = use_graph
    flow_fw, flow_bw, occ_fw, occ_bw = bi.forward_backward(l, r)
    assert flow_fw.shape == flow_bw.shape == (B, H, W, 2) and occ_fw.shape == occ_bw.shape == (B, H, W)
    assert occ_fw.dtype == torch.uint8 and occ_fw.is_cuda
    uni = _model(cuda, small, H, W, iters, B, volume_free)  # separate unidirectional model, same weights
    assert torch.equal(flow_fw, uni.forward(l, r)), "forward half differs from forward(l, r)"
    assert torch.equal(flow_bw, uni.forward(r, l)), "backward half differs from forward(r, l)"
    # the masks are the stand-alone kernel on the returned flows, bit for bit
    scale = 8.0 if small else 1.0
    ref_fw, ref_bw = _abi_consistency(flow_fw, flow_bw, scale)
    assert torch.equal(occ_fw, ref_fw) and torch.equal(occ_bw, ref_bw)
    assert set(torch.cat([occ_fw, occ_bw]).unique().tolist()) <= {0, 1, 2}
    # other thresholds are captured into a new graph
    _, _, occ2_fw, occ2_bw = bi.forward_backward(l, r, alpha1=0.05, alpha2=0.0)
    ref2_fw, ref2_bw = _abi_consistency(flow_fw, flow_bw, scale, 0.05, 0.0)
    assert torch.equal(occ2_fw, ref2_fw) and torch.equal(occ2_bw, ref2_bw)
    if use_graph:  # graph against eager
        bi.engine().use_graph = False
        eager = bi.forward_backward(l, r)
        assert torch.equal(eager[0], flow_fw) and torch.equal(eager[1], flow_bw) and torch.equal(eager[2], occ_fw)


def test_switching_entry_points_keeps_both_paths(cuda):
    """Alternating forward and forward_backward re-captures; each path computes what it computes alone, and the
    unidirectional launch count is unchanged."""
    from raft_b200 import synth
    H, W, iters = 64, 96, 2
    l, r = synth.make_batch(1, H, W)
    m = _model(cuda, False, H, W, iters)
    eng = m.engine()
    f0 = m.forward(l, r)
    n_uni = eng.launches_per_forward()
    fw, bw, occ_fw, _ = m.forward_backward(l, r)
    n_bi = eng.launches_per_forward()
    f1 = m.forward(l, r)
    assert eng.launches_per_forward() == n_uni and n_bi > n_uni
    assert torch.equal(f0, f1) and torch.equal(f0, fw)
    assert torch.equal(m.forward_backward(l, r)[3], _abi_consistency(fw, bw, 1.0)[1])


def _smooth_field(B, H, W, seed, amp):
    """Sum of random sinusoids (like synth.make_pair's motion), [B,H,W,2] fp32."""
    rng = np.random.default_rng(seed)
    ys, xs = np.meshgrid(np.arange(H, dtype=np.float64), np.arange(W, dtype=np.float64), indexing="ij")
    out = np.zeros((B, H, W, 2))
    for b in range(B):
        for c in range(2):
            for k in range(3):
                fx, fy, ph = rng.uniform(0.2, 1.0), rng.uniform(0.2, 1.0), rng.uniform(0, 2 * np.pi)
                out[b, ..., c] += amp / (k + 1) * np.sin(2 * np.pi * (fx * xs / W + fy * ys / H) + ph)
    return torch.from_numpy(out).float()


@pytest.mark.parametrize("scale", [1.0, 8.0])
def test_kernel_matches_fp64_oracle(cuda, scale):
    """Smooth forward field, backward = -forward plus a smooth disagreement of up to 2 px: every code is common.
    Codes equal the oracle's except at near-ties (|lhs - rhs| <= 1e-4 max(1, rhs), or t within 1e-4 px of the border),
    which stay under 0.1 % of the pixels."""
    B, H, W = 2, 67, 141
    fw = _smooth_field(B, H, W, 1, 6.0) / scale
    bw = (-fw + _smooth_field(B, H, W, 2, 1.0) / scale).contiguous()
    occ_fw, occ_bw = _abi_consistency(fw.to(cuda), bw.to(cuda), scale)
    ref_fw, ref_bw, m_fw, m_bw = fb_consistency(fw, bw, scale, 0.01, 0.5, return_margin=True)
    n = B * H * W
    for got, ref, (diff, rhs, border) in ((occ_fw.cpu(), ref_fw, m_fw), (occ_bw.cpu(), ref_bw, m_bw)):
        for code in (0, 1, 2):
            assert (ref == code).sum() > 0.02 * n, f"code {code} too rare to test: {(ref == code).sum()}"
        tie = (diff.abs() <= 1e-4 * rhs.clamp(min=1.0)) | (border.abs() <= 1e-4)
        bad = (got != ref) & ~tie
        assert not bad.any(), f"{int(bad.sum())} pixels differ from the oracle away from ties"
        assert tie.sum() < 1e-3 * n, int(tie.sum())


def test_kernel_handles_unaligned_mask_rows(cuda):
    """W = 7 (mask rows not 4-byte aligned: per-byte stores) and W = 1, against the oracle on translations."""
    for H, W in ((9, 7), (5, 1), (3, 12)):
        fw = torch.zeros(3, H, W, 2)
        fw[..., 0], fw[..., 1] = 1.5, -1.0
        bw = -fw
        bw[1] += 0.9  # |u + g|^2 = 1.62 >= 0.5 + ...: occluded wherever inside
        occ = _abi_consistency(fw.to(cuda), bw.to(cuda), 1.0)
        ref = fb_consistency(fw, bw)
        assert torch.equal(occ[0].cpu(), ref[0]) and torch.equal(occ[1].cpu(), ref[1]), (H, W)


def test_cli_bidirectional(cuda, tmp_path, monkeypatch):
    """--bidirectional writes the backward flow and the occlusion mask (PNG and .npy); the forward .npy is the one the
    CLI writes without the flag, byte for byte."""
    import cv2
    from raft_b200 import synth
    l, r = synth.make_batch(1, 60, 100)
    for name, img in (("a.png", l[0]), ("b.png", r[0])):
        cv2.imwrite(str(tmp_path / name), (img * 255).astype(np.uint8))
    np.savez(tmp_path / "w.npz", **synth.make_weights(False))
    spec = importlib.util.spec_from_file_location("infer_raft_cli_bidir", os.path.join(ROOT, "raft-tf_b200", "infer_raft.py"))
    cli = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(cli)
    monkeypatch.chdir(tmp_path)
    common = ["--im1", "a.png", "--im2", "b.png", "--load", "w.npz", "--iters", "2", "--keep-size"]
    assert cli.main(common + ["--npy", "plain.npy"]) == 0
    assert not os.path.exists("raft_flow_backward.png") and not os.path.exists("raft_occlusion.png")
    plain_png = open("raft_flow_raft-things.png", "rb").read()
    assert cli.main(common + ["--npy", "bi.npy", "--bidirectional"]) == 0
    assert open("plain.npy", "rb").read() == open("bi.npy", "rb").read()
    assert open("raft_flow_raft-things.png", "rb").read() == plain_png
    bw, occ = np.load("bi_backward.npy"), np.load("bi_occ.npy")
    assert bw.shape == (60, 100, 2) and bw.dtype == np.float32
    assert occ.shape == (2, 60, 100) and occ.dtype == np.uint8
    png = cv2.imread("raft_occlusion.png", cv2.IMREAD_UNCHANGED)
    assert png.shape == (60, 100) and np.array_equal(png, np.array([0, 255, 128], np.uint8)[occ[0]])
    assert cv2.imread("raft_flow_backward.png").shape == (60, 100, 3)
    a, b = cli.read_pair("a.png", "b.png", None)
    ref = _model(cuda, False, 60, 100, 2).forward(b, a)[0].cpu().numpy()
    assert np.array_equal(bw, ref)
