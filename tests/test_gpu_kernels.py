"""GPU parity tests of the individual kernels against the CPU oracle (all calls go through the C ABI).
Tolerances: lookup / sampler / grid are BIT-EXACT (same fp32 operation order as the oracle); GEMM-shaped
ops differ by fp32 summation order and the 2^-22 split-operand truncation -> relative 2e-5 of the
output scale; the final flow tolerance (1e-3 max-abs, BASELINE north_star) is in test_gpu_e2e.py."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import raft_oracle as O

pytestmark = pytest.mark.gpu


def _modes():
    from raft_b200 import capi
    return [("tc", capi.RB_MATH_TC), ("simt", capi.RB_MATH_SIMT)]


def _rand_pyramid(B, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(B * h * w, h >> l, w >> l, 1, generator=g) for l in range(4)]


def _coords(B, h, w, seed, spread=8.0, oob_frac=0.05):
    g = torch.Generator().manual_seed(seed)
    c = O.coords_grid(B, h, w) + (torch.rand(B, h, w, 2, generator=g) * 2 - 1) * spread
    m = torch.rand(B, h, w, 1, generator=g) < oob_frac
    far = (torch.rand(B, h, w, 2, generator=g) * 4 - 2) * torch.tensor([float(w), float(h)])
    c = torch.where(m, far, c)
    # exact integers, exact negatives in (-1,0), and exact borders must be present
    c[0, 0, 0] = torch.tensor([-0.75, -0.25])
    c[0, 0, 1] = torch.tensor([float(w - 1), float(h - 1)])
    c[0, 0, 2] = torch.tensor([3.0, 2.0])
    c[0, 0, 3] = torch.tensor([-1.0, -5.5])
    return c.contiguous()


def test_coords_grid(cuda):
    from networks.utils import coords_grid
    g = coords_grid(2, 5, 7, cuda)
    assert torch.equal(g.cpu(), O.coords_grid(2, 5, 7))


@pytest.mark.parametrize("B,h,w,r", [(1, 16, 32, 4), (2, 13, 27, 3), (1, 55, 128, 4), (1, 8, 8, 3), (1, 9, 17, 4)])
def test_lookup_bit_exact(cuda, B, h, w, r):
    """SampleCorr (model_utils.py:224-249) incl. odd pyramid dims, OOB / negative / integer coords."""
    from networks.model_utils import SampleCorr
    pyr = _rand_pyramid(B, h, w, 1234)
    coords = _coords(B, h, w, 5)
    ref = O.sample_corr(pyr, coords, radius=r)
    out = SampleCorr([p.to(cuda) for p in pyr], coords.to(cuda), radius=r).cpu()
    bad = (out != ref)
    assert not bad.any(), f"{int(bad.sum())} of {bad.numel()} taps differ; max abs diff {(out - ref).abs().max():.3e}"


def test_lookup_rounding_slack_outside_the_box(cuda):
    """fl(c + d) can round UP across an integer (c = 15.999999, d = +4 -> 20.0 while trunc(c - 4) + 8 = 19): the window then
    reaches one row / column beyond the (2r+2)^2 footprint.  Lookup v5 stages (2r+2) rows and takes a per-tap global-load
    path for such units; columns have the slack inside the 12-column box.  Must stay bit-exact."""
    from networks.model_utils import SampleCorr
    B, h, w, r = 1, 48, 64, 4
    pyr = _rand_pyramid(B, h, w, 77)
    coords = _coords(B, h, w, 3)
    below = lambda v: float(np.nextafter(np.float32(v), np.float32(0)))  # noqa: E731  largest fp32 < v
    k = 0
    for cy in (16.0, 32.0, 8.0):
        for cx in (16.0, 32.0, 10.5):
            coords[0, 5 + k // 8, 8 + k % 8] = torch.tensor([below(cx) if cx != 10.5 else cx, below(cy)])
            coords[0, 20 + k // 8, 8 + k % 8] = torch.tensor([below(cy), below(cx) if cx != 10.5 else 3.25])
            k += 1
    # the anomaly is really present: trunc(fl(c + 4)) - trunc(c - 4) == 9 for these coordinates
    c = torch.tensor(below(16.0))
    assert int(torch.trunc(c + 4.0)) - int(torch.trunc(c - 4.0)) == 9
    ref = O.sample_corr(pyr, coords, radius=r)
    out = SampleCorr([p.to(cuda) for p in pyr], coords.to(cuda), radius=r).cpu()
    assert torch.equal(out, ref), f"{int((out != ref).sum())} taps differ"


@pytest.mark.parametrize("B,h,w,C,r", [(1, 16, 32, 256, 4), (2, 17, 30, 128, 3), (1, 55, 128, 256, 4)])
def test_volume_free_lookup_matches_materialised_path(cuda, B, h, w, C, r):
    """F2 (SURVEY 8(f)): rb_corr_otf_lookup == SampleCorr(GetCorrPyramid(f1, f2)) up to the summation order / operand
    rounding of the dot products, and both agree with the fp64 oracle (model_utils.py:199-249)."""
    from raft_b200 import capi
    from networks.model_utils import GetCorrPyramid, SampleCorr
    g = torch.Generator().manual_seed(21)
    f1 = torch.randn(B, h, w, C, generator=g)
    f2 = torch.randn(B, h, w, C, generator=g)
    # in-image coordinates: far outside the image the reference's clamped-x1 weights grow like |x| and cancel (utils.py:84-98),
    # which amplifies the 1e-6 relative differences between the three evaluations of the dot products beyond any fixed bound
    gen = torch.Generator().manual_seed(17)
    coords = O.coords_grid(B, h, w) + (torch.rand(B, h, w, 2, generator=gen) * 2 - 1) * 5.0
    coords[..., 0].clamp_(0.0, w - 1.0)
    coords[..., 1].clamp_(0.0, h - 1.0)
    coords = coords.contiguous()
    ref = O.sample_corr(O.get_corr_pyramid(f1.double(), f2.double()), coords.double(), radius=r)
    f1d, f2d, cd = f1.to(cuda), f2.to(cuda), coords.to(cuda)
    mat = SampleCorr(GetCorrPyramid(f1d, f2d), cd, radius=r).cpu()
    lib = capi.lib
    wsb = capi.size_query(lib.rb_corr_otf_workspace_bytes, B, h, w, C)
    ws = torch.zeros(wsb, dtype=torch.uint8, device=cuda)
    out = torch.empty(B, h, w, 4 * (2 * r + 1) ** 2, device=cuda)
    capi.check(lib.rb_corr_otf_prepare(capi.ptr(f2d), capi.ptr(ws), wsb, B, h, w, C, capi.stream()))
    capi.check(lib.rb_corr_otf_lookup(capi.ptr(f1d), capi.ptr(f2d), capi.ptr(ws), capi.ptr(cd), capi.ptr(out), B, h, w, C, r,
                                      capi.stream()))
    out = out.cpu()
    scale = ref.abs().max().item()
    e_otf, e_mat, e_rel = (out.double() - ref).abs().max().item(), (mat.double() - ref).abs().max().item(), (out - mat).abs().max().item()
    print(f"\nvolume-free vs fp64 {e_otf:.2e}, materialised vs fp64 {e_mat:.2e}, volume-free vs materialised {e_rel:.2e}, scale {scale:.2f}")
    assert e_otf < 2e-4 * scale and e_mat < 2e-4 * scale and e_rel < 2e-4 * scale


def test_lookup_split_output_matches_fp32(cuda):
    """The fast path writes hi/lo fp16 planes; they must reconstruct the fp32 lookup to 2^-21 relative."""
    from raft_b200 import capi
    B, h, w, r = 1, 16, 32, 4
    pyr = _rand_pyramid(B, h, w, 7)
    coords = _coords(B, h, w, 9).to(cuda)
    buf = torch.cat([p.reshape(-1) for p in pyr] + [torch.zeros(64)]).to(cuda)
    ref = O.sample_corr(pyr, coords.cpu(), radius=r)
    lib = capi.lib
    wsb = capi.size_query(lib.rb_update_workspace_bytes, 0, B, h, w)
    ws = torch.zeros(wsb, dtype=torch.uint8, device=cuda)
    capi.check(lib.rb_update_lookup(0, capi.ptr(ws), capi.ptr(buf), capi.ptr(coords), B, h, w, capi.stream()))
    torch.cuda.synchronize()
    npix = B * h * w
    plane = (npix * 384 * 2 + 1023) // 1024 * 1024
    hi = ws[:npix * 384 * 2].view(torch.float16).view(npix, 384).float().cpu()
    lo = ws[plane:plane + npix * 384 * 2].view(torch.float16).view(npix, 384).float().cpu()
    rec = (hi + lo / 2048.0)[:, :324].reshape(B, h, w, 324)
    assert (hi[:, 324:] == 0).all() and (lo[:, 324:] == 0).all(), "channel padding must stay zero"
    err = (rec - ref).abs() / ref.abs().clamp_min(1e-2)
    assert err.max() < 2 ** -20, err.max()


def test_bilinear_sampler_general(cuda):
    from networks.utils import bilinear_sampler
    g = torch.Generator().manual_seed(3)
    img = torch.randn(6, 9, 11, 1, generator=g)
    coords = (torch.rand(6, 5, 4, 2, generator=g) * 16 - 3)
    ref = O.bilinear_sampler(img, coords)
    out = bilinear_sampler(img.to(cuda), coords.to(cuda)).cpu()
    assert torch.equal(out, ref)


@pytest.mark.parametrize("mode", ["tc", "simt"])
@pytest.mark.parametrize("B,h,w,C", [(1, 16, 32, 128), (2, 13, 27, 256), (1, 24, 40, 256)])
def test_corr_pyramid(cuda, mode, B, h, w, C):
    """GetCorrPyramid (model_utils.py:199-221): GEMM + /sqrt(C) + 3x VALID 2x2 average pooling."""
    from raft_b200 import capi
    from networks.model_utils import GetCorrPyramid
    g = torch.Generator().manual_seed(11)
    f1 = torch.randn(B, h, w, C, generator=g)
    f2 = torch.randn(B, h, w, C, generator=g)
    ref = O.get_corr_pyramid(f1.double(), f2.double())
    capi.check(capi.lib.rb_set_math_mode(dict(_modes())[mode]))
    try:
        pyr = GetCorrPyramid(f1.to(cuda), f2.to(cuda))
        torch.cuda.synchronize()
    finally:
        capi.lib.rb_set_math_mode(capi.RB_MATH_TC)
    scale = ref[0].abs().max().item()
    for l in range(4):
        assert pyr[l].shape == ref[l].shape
        err = (pyr[l].cpu().double() - ref[l]).abs().max().item()
        assert err < 2e-5 * scale, f"level {l}: max abs err {err:.3e} (scale {scale:.2f}, mode {mode})"


CONV_CASES = [
    # B, h, w, cin, cout, kh, kw   -- every filter shape of the update block + awkward tile geometries
    (1, 16, 32, 64, 64, 1, 1),
    (1, 16, 32, 324, 256, 1, 1),
    (1, 16, 32, 256, 192, 3, 3),
    (1, 16, 32, 128, 64, 3, 3),
    (1, 16, 32, 256, 126, 3, 3),
    (1, 16, 32, 384, 256, 1, 5),
    (1, 16, 32, 384, 128, 5, 1),
    (1, 16, 32, 256, 2, 3, 3),
    (1, 16, 32, 256, 576, 1, 1),
    (2, 13, 27, 242, 192, 3, 3),
    (1, 55, 128, 128, 96, 3, 3),
    (1, 8, 8, 64, 16, 3, 3),
    (3, 9, 120, 128, 128, 3, 3),
]


@pytest.mark.parametrize("mode", ["tc", "simt"])
@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: "x".join(map(str, c)))
def test_conv2d(cuda, mode, case):
    """tensorpack Conv2D(stride 1,'same')+bias+ReLU (A14) against torch fp64."""
    from raft_b200 import capi
    B, h, w, cin, cout, kh, kw = case
    g = torch.Generator().manual_seed(sum(case))
    x = torch.randn(B, h, w, cin, generator=g)
    W = torch.randn(kh, kw, cin, cout, generator=g) * (2.0 / (kh * kw * cin)) ** 0.5
    b = torch.randn(cout, generator=g) * 0.1
    ref = O.conv2d(x.double(), W.double(), b.double(), 1, torch.relu)
    lib = capi.lib
    xd = x.to(cuda)
    y = torch.full((B, h, w, cout), float("nan"), device=cuda)
    wsb = capi.size_query(lib.rb_conv2d_workspace_bytes, B, h, w, cin, cout, kh, kw)
    ws = torch.zeros(wsb, dtype=torch.uint8, device=cuda)
    Wn, bn = np.ascontiguousarray(W.numpy()), np.ascontiguousarray(b.numpy())
    capi.check(lib.rb_set_math_mode(dict(_modes())[mode]))
    try:
        capi.check(lib.rb_conv2d(capi.ptr(xd), Wn.ctypes.data, bn.ctypes.data, capi.ptr(y), B, h, w, cin, cout, kh, kw,
                                 1, capi.ptr(ws), wsb, capi.stream()))
        torch.cuda.synchronize()
    finally:
        lib.rb_set_math_mode(capi.RB_MATH_TC)
    yc = y.cpu().double()
    assert torch.isfinite(yc).all(), f"{int((~torch.isfinite(yc)).sum())} non-finite outputs (unwritten?)"
    err = (yc - ref).abs().max().item()
    scale = ref.abs().max().item()
    assert err < 2e-5 * max(scale, 1.0), f"max abs err {err:.3e} (scale {scale:.2f})"


@pytest.mark.parametrize("mode", ["tc", "simt"])
@pytest.mark.parametrize("case", [(2, 36, 52, 64, 96, 3), (1, 37, 51, 64, 96, 3), (2, 36, 52, 96, 128, 1), (1, 33, 47, 32, 64, 1),
                                  (1, 40, 56, 3, 64, 7), (1, 39, 57, 3, 32, 7), (1, 9, 300, 16, 16, 3)],
                         ids=lambda c: "x".join(map(str, c)))
def test_conv2d_stride2(cuda, mode, case):
    """tensorpack Conv2D(strides=2, 'same') as the encoders call it (model_utils.py:21,39,68,92): TF pads before = total/2
    (0|1 for even, 1|1 for odd sizes with k=3; 2|3 and 3|3 with k=7), taps through TMA element strides.  vs torch fp64."""
    from raft_b200 import capi
    B, h, w, cin, cout, k = case
    g = torch.Generator().manual_seed(sum(case))
    x = torch.randn(B, h, w, cin, generator=g)
    W = torch.randn(k, k, cin, cout, generator=g) * (2.0 / (k * k * cin)) ** 0.5
    b = torch.randn(cout, generator=g) * 0.1
    ref = O.conv2d(x.double(), W.double(), b.double(), 2, torch.relu)
    lib = capi.lib
    oh, ow = (h + 1) // 2, (w + 1) // 2
    assert ref.shape == (B, oh, ow, cout)
    y = torch.full((B, oh, ow, cout), float("nan"), device=cuda)
    wsb = capi.size_query(lib.rb_conv2d_workspace_bytes, B, h, w, cin, cout, k, k)
    ws = torch.zeros(wsb, dtype=torch.uint8, device=cuda)
    Wn, bn = np.ascontiguousarray(W.numpy()), np.ascontiguousarray(b.numpy())
    capi.check(lib.rb_set_math_mode(dict(_modes())[mode]))
    try:
        capi.check(lib.rb_conv2d_strided(capi.ptr(x.to(cuda)), Wn.ctypes.data, bn.ctypes.data, capi.ptr(y), B, h, w, cin, cout,
                                         k, k, 2, 1, capi.ptr(ws), wsb, capi.stream()))
        torch.cuda.synchronize()
    finally:
        lib.rb_set_math_mode(capi.RB_MATH_TC)
    yc = y.cpu().double()
    assert torch.isfinite(yc).all(), f"{int((~torch.isfinite(yc)).sum())} non-finite outputs (unwritten?)"
    err = (yc - ref).abs().max().item()
    assert err < 2e-5 * max(ref.abs().max().item(), 1.0), f"max abs err {err:.3e}"
    assert lib.rb_conv2d_strided(capi.ptr(y), Wn.ctypes.data, None, capi.ptr(y), B, h, w, cin, cout, k, k, 3, 0, capi.ptr(ws), wsb,
                                 capi.stream()) == -3  # RB_ERR_UNSUPPORTED: stride 3


# (1, 9, 6): grids narrower than the 8-pixel window of the tensor-core convf1 run flow_conv7_kernel beside the
# tensor-core convs
@pytest.mark.parametrize("B,h,w", [(2, 12, 20), (1, 9, 6)])
@pytest.mark.parametrize("mode", ["tc", "simt"])
@pytest.mark.parametrize("small", [False, True])
def test_update_block(cuda, mode, small, B, h, w):
    """BasicUpdateBlock / SmallUpdateBlock (model_utils.py:172-194): (net, mask, delta_flow)."""
    from raft_b200 import capi, synth
    from networks import model_utils as MU
    hid, ctx, r = (96, 64, 3) if small else (128, 128, 4)
    K = 4 * (2 * r + 1) ** 2
    p = synth.make_weights(small)
    g = torch.Generator().manual_seed(21)
    net = torch.tanh(torch.randn(B, h, w, hid, generator=g))
    inp = torch.relu(torch.randn(B, h, w, ctx, generator=g))
    corr = torch.randn(B, h, w, K, generator=g) * 3
    flow = torch.randn(B, h, w, 2, generator=g) * 2
    pt = {k: torch.from_numpy(v).double() for k, v in p.items()}
    if small:
        rn, rm, rd = O.small_update_block(net.double(), inp.double(), corr.double(), flow.double(), pt)
    else:
        rn, rm, rd = O.basic_update_block(net.double(), inp.double(), corr.double(), flow.double(), pt)
    MU.set_variables(p)
    capi.check(capi.lib.rb_set_math_mode(dict(_modes())[mode]))
    try:
        fn = MU.SmallUpdateBlock if small else MU.BasicUpdateBlock
        n2, m2, d2 = fn(net.to(cuda), inp.to(cuda), corr.to(cuda), flow.to(cuda), "update_block", hid)
        torch.cuda.synchronize()
    finally:
        capi.lib.rb_set_math_mode(capi.RB_MATH_TC)
    assert (n2.cpu().double() - rn).abs().max() < 5e-5, (n2.cpu().double() - rn).abs().max()
    assert (d2.cpu().double() - rd).abs().max() < 5e-5, (d2.cpu().double() - rd).abs().max()
    if not small:
        assert (m2.cpu().double() - rm).abs().max() < 1e-4, (m2.cpu().double() - rm).abs().max()
    else:
        assert m2 is None


def test_upsample_convex_and_upflow8(cuda):
    from types import SimpleNamespace
    from networks.RAFT import RAFT
    from networks.utils import upflow8
    g = torch.Generator().manual_seed(4)
    flow = torch.randn(2, 5, 7, 2, generator=g) * 3
    mask = torch.randn(2, 5, 7, 576, generator=g)
    ref = O.upsample_flow(flow.double(), mask.double())
    out = RAFT((40, 56, 3), SimpleNamespace(small=False)).upsample_flow(flow.to(cuda), mask.to(cuda)).cpu().double()
    assert (out - ref).abs().max() < 1e-4  # flow + grid - grid round trip costs ~1e-6 * 8
    ref8 = O.upflow8(flow)
    out8 = upflow8(flow.to(cuda)).cpu()
    assert (out8 - ref8).abs().max() < 1e-5


def test_error_paths_do_not_abort(cuda):
    from raft_b200 import capi
    lib = capi.lib
    t = torch.zeros(16, device=cuda)
    assert lib.rb_corr_lookup(capi.ptr(t), capi.ptr(t), capi.ptr(t), 1, 8, 8, 5, capi.stream()) == -3
    assert b"radius" in lib.rb_last_error()
    assert lib.rb_corr_build(None, None, None, 1, 8, 8, 256, None, 0, None) == -2


@pytest.mark.parametrize("mode", ["tc", "simt"])
@pytest.mark.parametrize("small,name,norm,out_dim,B,H,W", [
    (False, "fnet", "instance", 256, 2, 64, 96), (False, "cnet", "batch", 256, 1, 72, 104),
    (True, "fnet", "instance", 128, 2, 64, 96), (True, "cnet", "none", 160, 1, 72, 104),
    # odd sizes at every level: TF SAME pads 3|3 (stem) and 1|1 (3x3 s2) instead of 2|3 and 0|1
    (False, "cnet", "batch", 256, 2, 71, 99), (True, "fnet", "instance", 128, 1, 67, 85)])
def test_encoder(cuda, mode, small, name, norm, out_dim, B, H, W):
    """BasicEncoder / SmallEncoder (model_utils.py:61-105) on raft_b200's own kernels vs the fp64 oracle:
    asymmetric TF 'SAME' padding on the stride-2 convs, instance norm / folded batch norm / no norm."""
    from raft_b200 import capi, synth
    from raft_b200.encoders import CudaEncoder
    p = synth.make_weights(small)
    g = torch.Generator().manual_seed(31)
    img = torch.rand(B, H, W, 3, generator=g)
    pt = {k: torch.from_numpy(v).double() for k, v in p.items()}
    enc = O.small_encoder if small else O.basic_encoder
    ref = enc(2.0 * img.double() - 1.0, pt, name, norm)
    capi.check(capi.lib.rb_set_math_mode(dict(_modes())[mode]))
    try:
        out = CudaEncoder(p, name, small, norm, out_dim, cuda)(img.to(cuda))
        torch.cuda.synchronize()
    finally:
        capi.lib.rb_set_math_mode(capi.RB_MATH_TC)
    assert out.shape == ref.shape
    err = (out.cpu().double() - ref).abs().max().item()
    assert err < 1e-4 * max(ref.abs().max().item(), 1.0), f"max abs err {err:.3e} (scale {ref.abs().max():.2f})"
