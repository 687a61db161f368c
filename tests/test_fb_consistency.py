"""Forward-backward consistency check (F5) without a GPU: the fp64 oracle on constructed flow fields, and the argument
checks of rb_flow_consistency (they run before any CUDA call)."""
import ctypes
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))  # fb_oracle.py sits beside the tests
from fb_oracle import fb_consistency  # noqa: E402


def _const(B, H, W, dx, dy):
    f = torch.empty(B, H, W, 2, dtype=torch.float32)
    f[..., 0], f[..., 1] = dx, dy
    return f


def _leaves(H, W, ux, uy):
    ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float64), torch.arange(W, dtype=torch.float64), indexing="ij")
    tx, ty = xs + ux, ys + uy
    return (tx < 0) | (tx > W - 1) | (ty < 0) | (ty > H - 1)


@pytest.mark.parametrize("dx,dy", [(3.0, -2.0), (-2.5, 1.25), (0.0, 0.0), (7.0, 4.5)])
def test_translation_is_consistent_inside_and_leaves_outside(dx, dy):
    B, H, W = 2, 13, 21
    occ_fw, occ_bw = fb_consistency(_const(B, H, W, dx, dy), _const(B, H, W, -dx, -dy))
    assert occ_fw.dtype == torch.uint8 and occ_fw.shape == (B, H, W)
    for occ, s in ((occ_fw, 1.0), (occ_bw, -1.0)):
        out = _leaves(H, W, s * dx, s * dy)
        assert torch.equal(occ, torch.where(out, 2, 0).to(torch.uint8).expand(B, H, W))


def test_scale_multiplies_the_displacement():
    """scale = 8 on a flow of d/8 px is the check of a flow of d px; scale = 1 on the same d/8 flow is a different one."""
    B, H, W, dx, dy = 1, 17, 40, 12.0, -5.0
    fw, bw = _const(B, H, W, dx, dy), _const(B, H, W, -dx, -dy)
    want = fb_consistency(fw, bw)
    got = fb_consistency(fw / 8, bw / 8, scale=8.0)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    assert (want[0] == 2).sum() > (fb_consistency(fw / 8, bw / 8)[0] == 2).sum()
    # a backward flow off by 1 unit: |u + g|^2 = 1 < alpha2 = 2 at scale 1, but 64 at scale 8
    bw1 = _const(B, H, W, -dx / 8 + 1.0, -dy / 8)
    at1 = fb_consistency(fw / 8, bw1, alpha2=2.0)[0]
    at8 = fb_consistency(fw / 8, bw1, scale=8.0, alpha2=2.0)[0]
    assert set(at1.unique().tolist()) <= {0, 2} and (at1 == 0).any()
    assert set(at8.unique().tolist()) <= {1, 2} and (at8 == 1).any()


def test_known_disagreement_is_occluded():
    """Backward flow zeroed on a block: forward pixels whose target's whole bilinear support lies in the block see
    g = 0, |u|^2 = 25 >= 0.01 * 25 + 0.5 -> 1; targets whose support avoids the block stay 0."""
    B, H, W, dx, dy = 1, 30, 40, 3.0, 4.0
    fw, bw = _const(B, H, W, dx, dy), _const(B, H, W, -dx, -dy)
    bw[:, 10:20, 15:25] = 0.0
    occ_fw, occ_bw = fb_consistency(fw, bw)
    ys, xs = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    tx, ty = xs + 3, ys + 4  # integer targets: the support is the target pixel itself (zero weight on the others)
    in_block = (ty >= 10) & (ty < 20) & (tx >= 15) & (tx < 25)
    assert (occ_fw[0][in_block] == 1).all() and in_block.sum() == 100
    inside = (tx <= W - 1) & (ty <= H - 1)
    assert (occ_fw[0][inside & ~in_block] == 0).all()
    assert (occ_fw[0][~inside] == 2).all()
    # the zero-flow block in the backward direction stays inside, and the forward flow at its (unmoved) target is
    # (3, 4): |0 + (3,4)|^2 = 25 -> occluded there too
    assert (occ_bw[0, 10:20, 15:25] == 1).all()
    # a fractional target half in the block: g = 0.5 * (-3,-4), |u + g|^2 = 5 >= 0.01 (22.25 + 6.25) + 0.5 -> 1
    half = fb_consistency(_const(B, H, W, 2.5, 4.0), bw)[0]
    assert half[0, 8, 12] == 1  # t = (14.5, 12): corners x = 14 (outside the block) and 15 (inside)


def test_margins_locate_the_decision():
    B, H, W = 1, 9, 11
    fw, bw = _const(B, H, W, 1.0, 0.0), _const(B, H, W, -1.0, 0.0)
    occ_fw, _, (diff, rhs, border), _ = fb_consistency(fw, bw, return_margin=True)
    inside = occ_fw[0] != 2
    assert torch.allclose(diff[0][inside], torch.tensor(-(0.01 * 2 + 0.5), dtype=torch.float64))
    assert torch.allclose(rhs[0][inside], torch.tensor(0.52, dtype=torch.float64))
    assert (border[0][:, W - 2] == 0).all() and (border[0][:, W - 1] < 0).all()  # t = W - 1 is on the border, inside


def _abi():
    from raft_b200 import capi
    buf = (ctypes.c_double * 64)()  # 8-byte aligned host memory: the checks never dereference it
    return capi.lib, ctypes.cast(buf, ctypes.c_void_p), buf


@pytest.mark.parametrize("null", range(4))
def test_abi_rejects_null_pointers(null):
    lib, p, _keep = _abi()
    ptrs = [p, p, p, p]
    ptrs[null] = None
    assert lib.rb_flow_consistency(*ptrs, 1, 8, 8, 1.0, 0.01, 0.5, None) == -2  # RB_ERR_BAD_ARG
    assert b"null pointer" in lib.rb_last_error()


@pytest.mark.parametrize("B,H,W", [(0, 8, 8), (1, 0, 8), (1, 8, 0), (-1, 8, 8), (1, -3, 8), (1, 8, -5)])
def test_abi_rejects_bad_shapes(B, H, W):
    lib, p, _keep = _abi()
    assert lib.rb_flow_consistency(p, p, p, p, B, H, W, 1.0, 0.01, 0.5, None) == -1  # RB_ERR_BAD_SHAPE
    assert b"bad shape" in lib.rb_last_error()


@pytest.mark.parametrize("scale,a1,a2,what", [(1.0, -0.01, 0.5, b"alpha"), (1.0, 0.01, -0.5, b"alpha"),
                                               (1.0, float("nan"), 0.5, b"alpha"), (0.0, 0.01, 0.5, b"scale"),
                                               (-8.0, 0.01, 0.5, b"scale")])
def test_abi_rejects_bad_parameters(scale, a1, a2, what):
    lib, p, _keep = _abi()
    assert lib.rb_flow_consistency(p, p, p, p, 1, 8, 8, scale, a1, a2, None) == -2  # RB_ERR_BAD_ARG
    assert what in lib.rb_last_error()


def test_abi_rejects_misaligned_flow():
    lib, p, _keep = _abi()
    q = ctypes.c_void_p(p.value + 4)
    assert lib.rb_flow_consistency(q, p, p, p, 1, 8, 8, 1.0, 0.01, 0.5, None) == -2
    assert b"aligned" in lib.rb_last_error()
