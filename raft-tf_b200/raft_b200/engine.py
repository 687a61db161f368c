"""Host-side orchestration of one RAFT forward pass on one GPU.

rb_encoder_forward x2 (fnet on both frames, cnet on a forked stream; csrc/encoder.cu) -> rb_corr_build ->
rb_update_set_state_cnet -> rb_raft_iterate (lookup + update block per iteration) -> rb_upsample_convex /
rb_upflow8, all replayed from ONE CUDA graph.  Mirrors RAFT.network_graph (networks/RAFT.py:78-109).

forward_backward runs both directions as one batch of 2B pairs ([l->r | r->l]) through the same kernels and adds the
forward-backward consistency check (rb_flow_consistency) to the graph.
"""
from __future__ import annotations

import os
from typing import Dict, Optional

import numpy as np
import torch

from . import capi
from .encoders import CudaEncoder
from .weights import pack_update_block


class RaftEngine:
    def __init__(self, params: Dict[str, np.ndarray], small: bool = False, iters: int = 20,
                 device: Optional[torch.device] = None, use_graph: bool = True, math_mode: int = capi.RB_MATH_TC,
                 volume_free: Optional[bool] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("raft_b200 needs a CUDA device (no CPU fallback)")
        self.device = torch.device(device if device is not None else "cuda:0")
        self.small, self.iters = bool(small), int(iters)
        self.hidden, self.ctx, self.radius, self.fdim = (96, 64, 3, 128) if small else (128, 128, 4, 256)
        self.use_graph = use_graph and not os.environ.get("RAFT_B200_NO_GRAPH")
        # F2 (opt-in): no materialised correlation volume -- every iteration evaluates the dot products its taps touch
        # straight from the feature maps (rb_update_lookup_otf).  Saves 4*N^2*1.33 bytes per pair (261 MB at 440x1024),
        # costs ~100 k extra FMA per pixel and iteration on the CUDA cores; same flow up to fp32 summation order.
        self.volume_free = bool(os.environ.get("RAFT_B200_VOLUME_FREE")) if volume_free is None else bool(volume_free)
        self.math_mode = math_mode
        # pixels per flow unit for the consistency check: raft-small's upflow8 keeps the reference's missing x8
        # (networks/utils.py:105-111, SURVEY fact 8); the returned flows are left as they are
        self.flow_scale = 8.0 if small else 1.0
        cnorm = "none" if small else "batch"
        with torch.cuda.device(self.device):
            self.fnet = CudaEncoder(params, "fnet", small, "instance", self.fdim, self.device)
            self.cnet = CudaEncoder(params, "cnet", small, cnorm, self.hidden + self.ctx, self.device)
            self.blob = pack_update_block(params, small, self.device)
        self._shape = None
        self._graph = None
        self._enc_stream = None   # forked stream of the context encoder (encode())
        self._capture_stream = None  # CUDA-graph capture stream on this engine's device (run())
        self._cnet_pending = False
        self._range_checked = set()  # directions (bidirectional flag) whose buffers passed the fp16-range check
        self._alphas = None  # thresholds of the consistency check captured in the bidirectional graph

    # ---- buffers -------------------------------------------------------------------------------
    def _ensure(self, B: int, H: int, W: int, u8: bool = False, bidir: bool = False):
        """Buffers for B frame pairs of H x W pixels.  H, W need not be multiples of 8: frames are replicate-padded
        to (Hp, Wp) by rb_frames_prepare (upstream InputPadder 'sintel' split, SURVEY 8(d)) and the flow is cropped
        back by the upsampling kernel -- the reference itself cannot run such shapes (SURVEY fact 6).

        bidir: the hot path runs at NB = 2B pairs, [left->right | right->left]; the feature maps are stored as
        [fA | fB | fA] so that fmap1 = [fA | fB] and fmap2 = [fB | fA] are contiguous views.  The buffers and the graph
        serve one mode: alternating forward and forward_backward reallocates and re-captures on every switch."""
        if self._shape == (B, H, W, u8, bidir):
            return
        NB = 2 * B if bidir else B
        ph, pw = (-H) % 8, (-W) % 8
        self.pad = (ph // 2, ph - ph // 2, pw // 2, pw - pw // 2)  # top, bottom, left, right
        Hp, Wp = H + ph, W + pw
        h, w, s = Hp // 8, Wp // 8, int(self.small)
        d = self.device
        lib = capi.lib
        self.h, self.w, self.Hp, self.Wp = h, w, Hp, Wp
        if self.volume_free:
            self.pyr_bytes, self.pyramid = 0, None
            self.cws_bytes = capi.size_query(lib.rb_corr_otf_workspace_bytes, NB, h, w, self.fdim)  # pooled fmap2, levels 1..3
        else:
            self.pyr_bytes = capi.size_query(lib.rb_corr_pyramid_bytes, NB, h, w)
            self.pyramid = torch.empty(self.pyr_bytes // 4, dtype=torch.float32, device=d)
            self.cws_bytes = capi.size_query(lib.rb_corr_workspace_bytes, NB, h, w, self.fdim)
        self.corr_ws = torch.zeros(self.cws_bytes, dtype=torch.uint8, device=d)
        self.ws_bytes = capi.size_query(lib.rb_update_workspace_bytes, s, NB, h, w)
        self.ws = torch.zeros(self.ws_bytes, dtype=torch.uint8, device=d)  # zero fill = channel padding
        self.coords1 = torch.empty(NB, h, w, 2, dtype=torch.float32, device=d)
        self.mask = None if self.small else torch.empty(NB, h, w, 576, dtype=torch.float32, device=d)
        self.flow_up = torch.empty(NB, H, W, 2, dtype=torch.float32, device=d)
        self.occ = torch.empty(NB, H, W, dtype=torch.uint8, device=d) if bidir else None
        self.fmaps = torch.empty(B + NB, h, w, self.fdim, dtype=torch.float32, device=d)
        self.fmap1, self.fmap2 = self.fmaps[:NB], self.fmaps[B:]
        self.cmap = torch.empty(NB, h, w, self.hidden + self.ctx, dtype=torch.float32, device=d)
        self.images = torch.empty(2 * B, Hp, Wp, 3, dtype=torch.float32, device=d)  # [left | right], [0,1], padded
        # staging buffer of the raw frames (uint8 or unpadded fp32); fp32 frames that need no padding go straight
        # into self.images
        self.staged = bool(u8 or ph or pw)
        self.raw = torch.empty(2 * B, H, W, 3, dtype=torch.uint8 if u8 else torch.float32, device=d) if self.staged else None
        self.nb = NB
        self._shape = (B, H, W, u8, bidir)
        self._graph = None

    # ---- stages --------------------------------------------------------------------------------
    def encode(self, defer_join: bool = False):
        """RAFT.py:53-59,79-87 on self.images = [left | right]: 2x-1, fnet(left), fnet(right), cnet(left) (bidirectional:
        cnet(right) too, and fmaps becomes [fA | fB | fA]).

        The context encoder is independent of the feature encoder (RAFT.py:79-87) and both are chains of ~50 small
        kernels at 1/4 and 1/8 resolution: cnet runs on a forked stream beside fnet (a fork/join that is captured into
        the CUDA graph like the flow branch of the update block).  With defer_join the caller joins (`_join_cnet`)
        where cmap is first needed -- after the correlation volume, which only needs the feature maps."""
        B, H, W, u8, bidir = self._shape
        capi.check(capi.lib.rb_set_math_mode(self.math_mode))  # per-thread library state: set before ANY kernel of ours
        if self.staged:  # F3: u8 -> fp32 /255 and replicate padding in one pass (csrc/frames.cu)
            capi.check(capi.lib.rb_frames_prepare(capi.ptr(self.raw), int(u8), capi.ptr(self.images), 2 * B, H, W,
                                                  *self.pad, capi.stream()))
        main = torch.cuda.current_stream(self.device)
        if self._enc_stream is None:
            self._enc_stream = torch.cuda.Stream(device=self.device)
        side = self._enc_stream
        side.wait_stream(main)  # fork: the frames are in place
        with torch.cuda.stream(side):
            self.cnet(self.images[:self.nb], out=self.cmap)  # bidirectional: context of both directions' first frame
        self.fnet(self.images, out=self.fmaps[:2 * B])
        if bidir:
            self.fmaps[2 * B:].copy_(self.fmaps[:B])  # [fA | fB] -> [fA | fB | fA]: a device-to-device memcpy, no kernel
        self._cnet_pending = True
        if not defer_join:
            self._join_cnet()

    def _join_cnet(self):
        if self._cnet_pending:
            torch.cuda.current_stream(self.device).wait_stream(self._enc_stream)
            self._cnet_pending = False

    def _hot_path(self):
        """corr build + iterations + upsampling: hand-written kernels only (graph-capturable)."""
        B, H, W, _, bidir = self._shape
        NB = self.nb
        h, w, s, lib, st = self.h, self.w, int(self.small), capi.lib, capi.stream()
        capi.check(lib.rb_set_math_mode(self.math_mode))
        if self.volume_free:
            capi.check(lib.rb_corr_otf_prepare(capi.ptr(self.fmap2), capi.ptr(self.corr_ws), self.cws_bytes, NB, h, w, self.fdim, st))
        else:
            capi.check(lib.rb_corr_build(capi.ptr(self.fmap1), capi.ptr(self.fmap2), capi.ptr(self.pyramid), NB, h, w,
                                         self.fdim, capi.ptr(self.corr_ws), self.cws_bytes, st))
        self._join_cnet()  # cmap (context encoder, forked stream) is first needed here
        capi.check(lib.rb_update_set_state_cnet(s, capi.ptr(self.blob), capi.ptr(self.ws), capi.ptr(self.cmap), NB, h, w, st))
        capi.check(lib.rb_coords_grid(capi.ptr(self.coords1), NB, h, w, st))
        if self.volume_free:  # RAFT.py:91-102 with the lookup evaluated on the fly
            for it in range(self.iters):
                capi.check(lib.rb_update_lookup_otf(s, capi.ptr(self.ws), capi.ptr(self.fmap1), capi.ptr(self.fmap2),
                                                    capi.ptr(self.corr_ws), capi.ptr(self.coords1), NB, h, w, self.fdim, st))
                mask = self.mask if (it == self.iters - 1 and not self.small) else None
                capi.check(lib.rb_update_step(s, capi.ptr(self.blob), capi.ptr(self.ws), capi.ptr(self.coords1), None,
                                              capi.ptr(mask), NB, h, w, st))
        else:
            capi.check(lib.rb_raft_iterate(s, capi.ptr(self.blob), capi.ptr(self.ws), capi.ptr(self.pyramid),
                                           capi.ptr(self.coords1), capi.ptr(self.mask), NB, h, w, self.iters, st))
        top, left = self.pad[0], self.pad[2]  # crop the padding away while upsampling
        if self.small:
            capi.check(lib.rb_upflow8_crop(capi.ptr(self.coords1), capi.ptr(self.flow_up), NB, h, w, 1.0, top, left, H, W, st))
        else:
            capi.check(lib.rb_upsample_convex_crop(capi.ptr(self.coords1), capi.ptr(self.mask), capi.ptr(self.flow_up),
                                                   NB, h, w, top, left, H, W, st))
        if bidir:  # both directions in one launch: occ[:B] checks flow_up[:B] against flow_up[B:], occ[B:] the reverse
            a1, a2 = self._alphas
            capi.check(lib.rb_flow_consistency(capi.ptr(self.flow_up[:B]), capi.ptr(self.flow_up[B:]), capi.ptr(self.occ[:B]),
                                               capi.ptr(self.occ[B:]), B, H, W, self.flow_scale, a1, a2, st))

    def _all(self):
        self.encode(defer_join=True)
        self._hot_path()

    def launches_per_forward(self) -> int:
        """Number of raft_b200 kernels one forward pass launches (counted by the library)."""
        capi.lib.rb_launch_count_reset()
        with torch.cuda.device(self.device):
            self._all()
            torch.cuda.synchronize()
        return int(capi.lib.rb_launch_count())

    def run(self):
        """encoders + hot path on self.images, replayed from one CUDA graph."""
        if not self.use_graph:
            self._all()
            return
        if self._graph is None:
            self._all()  # warm-up: function attributes, tensor-map cache
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            # torch.cuda.graph's default capture stream is a process-wide singleton on whichever device used it first, and
            # entering it switches the current device to THAT device: an engine on another device of the same process
            # would record its kernels there (illegal address at replay).  Capture on a stream of this engine's device.
            if self._capture_stream is None:
                self._capture_stream = torch.cuda.Stream(device=self.device)
            with torch.cuda.graph(g, stream=self._capture_stream):
                self._all()
            self._graph = g
        self._graph.replay()

    def _submit(self, left: torch.Tensor, right: torch.Tensor, bidir: bool):
        assert left.shape == right.shape and left.dim() == 4 and left.shape[-1] == 3 and left.dtype == right.dtype
        u8 = left.dtype == torch.uint8
        assert u8 or left.dtype == torch.float32, left.dtype
        with torch.cuda.device(self.device):
            B = left.shape[0]
            self._ensure(B, left.shape[1], left.shape[2], u8, bidir)
            dst = self.raw if self.staged else self.images
            dst[:B].copy_(left, non_blocking=True)  # H2D when the caller hands pinned host tensors
            dst[B:].copy_(right, non_blocking=True)
            self.run()
            if bidir not in self._range_checked:
                self._check_range(bidir)

    @torch.no_grad()
    def forward(self, left: torch.Tensor, right: torch.Tensor) -> torch.Tensor:
        """left/right: [B,H,W,3] frames, BGR like the reference: fp32 in [0,1] (RAFT.inputs(), RAFT.py:45-51) or
        uint8 in [0,255] (what cv2.imdecode yields, test_dataflow.py:56-61; the /255 then happens on the GPU).  Host
        (ideally pinned) or CUDA tensors; any H, W >= 8.  Returns the [B,H,W,2] flow -- the engine-owned buffer itself,
        overwritten by the next call (networks.RAFT.RAFT.forward hands out a copy)."""
        self._submit(left, right, False)
        return self.flow_up

    @torch.no_grad()
    def forward_backward(self, left: torch.Tensor, right: torch.Tensor, alpha1: float = 0.01, alpha2: float = 0.5):
        """Flow in both directions and their forward-backward consistency, from one graph: frames as for forward.
        Returns the engine-owned flow_up [2B,H,W,2] (left->right for the first B, right->left for the last B) and
        occ [2B,H,W] uint8 in the same order: 0 consistent, 1 occluded (the directions disagree:
        |u + g|^2 >= alpha1 (|u|^2 + |g|^2) + alpha2), 2 the displacement leaves the frame.  Each half of flow_up equals
        the corresponding forward() call bit for bit (a batch never mixes samples, DESIGN.md section 4).  The thresholds
        are captured in the graph: changing them re-captures."""
        alphas = (float(alpha1), float(alpha2))
        if alphas != self._alphas:
            self._alphas, self._graph = alphas, None
        self._submit(left, right, True)
        return self.flow_up, self.occ

    def _check_range(self, bidir: bool = False):
        """Once per engine and direction mode: the split-operand format (fp16 hi/lo planes) saturates beyond 65504.
        The fp32 tensors at the boundary of that path are the feature maps, the context map and the correlation volume;
        a checkpoint that drives them (or the result) out of range must fail loudly, not return a plausible-looking
        wrong flow.  The bidirectional buffers add the context map of the right frames and the reverse volume."""
        self._range_checked.add(bidir)
        if os.environ.get("RAFT_B200_NO_RANGE_CHECK"):
            return
        vol = self.pyramid[:self.pyr_bytes // 4 - 64].abs().max() if self.pyramid is not None else self.fmaps.new_zeros(())
        stats = torch.stack([self.fmaps.abs().max(), self.cmap.abs().max(), vol, self.flow_up.abs().max()]).tolist()
        names = ("feature maps", "context map", "correlation volume", "flow")
        for n, v in zip(names, stats):
            if not np.isfinite(v) or (n != "flow" and v > 6.0e4):
                raise capi.RaftB200Error(f"raft_b200: {n} reach |x|max = {v:.3g}: outside the fp16 range of the "
                                         "split-operand tensor-core path (csrc/common.cuh)")

    def lowres_flow(self) -> torch.Tensor:
        g = torch.stack(torch.meshgrid(torch.arange(self.w, device=self.device),
                                       torch.arange(self.h, device=self.device), indexing="xy"), -1).float()
        return self.coords1 - g[None]
