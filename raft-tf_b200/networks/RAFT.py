"""Drop-in mirror of the reference's ``networks/RAFT.py``: same class name, constructor signature
``RAFT(image_shape, args)`` (only ``args.small`` is read, RAFT.py:37), same attributes, same method
names.  The TF graph is replaced by raft_b200's CUDA engine; ``build_graph`` keeps the reference's
contract (returns 0.0 and publishes the result under the name ``flow_result``, RAFT.py:136-141) and
``forward`` is the direct call.  Extensions over the reference (which hard-codes them, SURVEY fact
5): ``iters``, ``batch`` and the image shape are honoured as parameters; inputs whose H/W are not
multiples of 8 are replicate-padded and the flow cropped back (the reference itself cannot run such
shapes, SURVEY fact 6)."""
import numpy as np
import torch

from networks import model_utils
from networks.model_utils import GetCorrPyramid, SampleCorr, BasicUpdateBlock, SmallUpdateBlock  # noqa: F401
from networks.utils import coords_grid, upflow8  # noqa: F401
from raft_b200 import capi
from raft_b200.engine import RaftEngine
from raft_b200.weights import load_npz


class RAFT(object):
    weight_decay = 1e-5          # vestigial in the reference too (RAFT.py:14)
    data_format = 'NHWC'

    def __init__(self, image_shape, args, iters=20, batch=1, device=None, volume_free=None):
        self.dropout = 0.0
        self.corr_radius = 4
        self.hidden_dim = 128
        self.context_dim = 128
        self.mode = 'test'
        self.iters = iters
        self.image_shape = image_shape
        self.batch = batch
        self.small = bool(getattr(args, 'small', False))
        if self.small:
            self.hidden_dim = 96
            self.context_dim = 64
            self.corr_radius = 3
        self.device = torch.device(device if device is not None else 'cuda:0')
        self.volume_free = volume_free  # extension (SURVEY 8(f) F2): None = RAFT_B200_VOLUME_FREE env, default off
        self.flow_result = None
        self._engine = None
        self._params = None

    # -- reference surface ------------------------------------------------------------------------
    def inputs(self):
        """RAFT.py:45-51: two [batch,H,W,3] fp32 inputs in [0,1] named input_left / input_right."""
        shp = (self.batch, self.image_shape[0], self.image_shape[1], self.image_shape[2])
        return [('input_left', shp, np.float32), ('input_right', shp, np.float32)]

    def input_preprocess(self, input_left, input_right):
        return 2.0 * input_left - 1.0, 2.0 * input_right - 1.0

    def initialize_flow(self, image):
        b, H, W = image.shape[0], image.shape[1], image.shape[2]
        return coords_grid(b, H // 8, W // 8, image.device), coords_grid(b, H // 8, W // 8, image.device)

    def upsample_flow(self, flow, mask):
        """RAFT.py:119-134 (convex 8x upsampling)."""
        b, h, w, _ = flow.shape
        coords1 = (flow + coords_grid(b, h, w, flow.device)).contiguous()
        out = torch.empty(b, 8 * h, 8 * w, 2, dtype=torch.float32, device=flow.device)
        with torch.cuda.device(flow.device):
            capi.check(capi.lib.rb_upsample_convex(capi.ptr(coords1), capi.ptr(mask.contiguous().float()),
                                                   capi.ptr(out), b, h, w, capi.stream()))
        return out

    def build_graph(self, input_left, input_right):
        self.flow_result = self.forward(input_left, input_right)
        return 0.0

    # -- weights (tensorpack get_model_loader(npz), infer_raft.py:77) ---------------------------
    def load(self, npz_or_params):
        self._params = load_npz(npz_or_params) if isinstance(npz_or_params, str) else dict(npz_or_params)
        model_utils.set_variables(self._params)
        self._engine = None
        return self

    def engine(self):
        if self._engine is None:
            if self._params is None:
                raise RuntimeError("RAFT.load(<npz>) must be called before inference")
            self._engine = RaftEngine(self._params, small=self.small, iters=self.iters, device=self.device,
                                      volume_free=self.volume_free)
        return self._engine

    # -- inference ---------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, input_left, input_right):
        """[B,H,W,3] frames, BGR like the reference -- fp32 in [0,1] (the reference's placeholders, RAFT.py:45-51) or
        uint8 in [0,255] (extension: the /255 of test_dataflow.py:96-97 then runs on the GPU); numpy or torch, host or
        CUDA -> [B,H,W,2] torch CUDA flow (a fresh tensor per call, like a session.run result).  H, W that are not
        multiples of 8 are replicate-padded and the flow cropped back, both inside the engine's own kernels."""
        flow = self.engine().forward(_as_frames(input_left), _as_frames(input_right))
        return flow.clone()

    @torch.no_grad()
    def forward_backward(self, input_left, input_right, alpha1=0.01, alpha2=0.5):
        """Extension: the flow in both directions and the forward-backward consistency masks, from one CUDA graph that
        runs the two directions as one batch (the feature maps of each frame are computed once).  Frames as for
        ``forward``.  Returns fresh CUDA tensors ``(flow_fw, flow_bw, occ_fw, occ_bw)``: flow_fw == forward(left, right)
        and flow_bw == forward(right, left) bit for bit, [B,H,W,2]; occ_* [B,H,W] uint8 with 0 = consistent,
        1 = occluded (|u + g|^2 >= alpha1 (|u|^2 + |g|^2) + alpha2, u the displacement at p and g the other direction's
        flow sampled bilinearly at p + u, Sundaram et al. 2010 / UnFlow), 2 = p + u leaves the frame.  Displacements are
        in full-resolution pixels: raft-small's flow, which keeps the reference's missing x8 of upflow8, is scaled by 8
        for the check only."""
        flow, occ = self.engine().forward_backward(_as_frames(input_left), _as_frames(input_right), alpha1, alpha2)
        B = flow.shape[0] // 2
        return flow[:B].clone(), flow[B:].clone(), occ[:B].clone(), occ[B:].clone()


def _as_frames(x):
    t = torch.as_tensor(x)
    return t if t.dtype == torch.uint8 else t.to(torch.float32)
