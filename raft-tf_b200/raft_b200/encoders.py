"""Feature / context encoders (networks/model_utils.py:6-105) on raft_b200's own kernels (csrc/encoder.cu).

Exact TF semantics: asymmetric 'SAME' padding on the stride-2 convs, instance norm without affine, BatchNorm with EMA
statistics.  Frames go in and feature maps come out NHWC, like the reference.
"""
from __future__ import annotations

from typing import Dict

import numpy as np
import torch


class CudaEncoder:
    """BasicEncoder (things) / SmallEncoder (small) with weights keyed like the reference npz: every conv runs on the
    tcgen05 implicit-GEMM kernel of the update block (split fp16 operands), instance norm as a fused stats/apply pass,
    batch norm folded into the weights."""

    NORMS = {"none": 0, "instance": 1, "batch": 2}

    def __init__(self, params: Dict[str, np.ndarray], name: str, small: bool, norm_fn: str, out_dim: int, device):
        import ctypes as C
        from . import capi
        self.capi, self.small, self.norm, self.out_dim = capi, int(bool(small)), self.NORMS[norm_fn], int(out_dim)
        self.device = torch.device(device)
        lib = capi.lib
        n = lib.rb_encoder_num_convs(self.small)
        Ws, bs, bns, keep = (C.c_void_p * n)(), (C.c_void_p * n)(), (C.c_void_p * n)(), []
        for i in range(n):
            cname = f"{name}/{lib.rb_encoder_conv_name(self.small, i).decode()}"
            nname = lib.rb_encoder_norm_name(self.small, i).decode()
            k, s, ci, co = C.c_int(), C.c_int(), C.c_int(), C.c_int()
            capi.check(lib.rb_encoder_conv_shape(self.small, i, self.out_dim, C.byref(k), C.byref(s), C.byref(ci), C.byref(co)))
            W = np.ascontiguousarray(params[cname + "/W"], dtype=np.float32)
            b = np.ascontiguousarray(params[cname + "/b"], dtype=np.float32)
            want = (k.value, k.value, ci.value, co.value)
            if tuple(W.shape) != want:
                raise ValueError(f"{cname}: expected W{want}, got {tuple(W.shape)}")
            keep += [W, b]
            Ws[i], bs[i] = W.ctypes.data, b.ctypes.data
            if self.norm == 2 and nname:
                sc = f"{name}/{nname}"
                bn = np.ascontiguousarray(np.concatenate([params[sc + "/gamma"], params[sc + "/beta"], params[sc + "/mean/EMA"],
                                                          params[sc + "/variance/EMA"]]), dtype=np.float32)
                keep.append(bn)
                bns[i] = bn.ctypes.data
        nbytes = capi.size_query(lib.rb_encoder_weights_bytes, self.small, self.out_dim)
        self.blob = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            capi.check(lib.rb_encoder_weights_pack(self.small, self.norm, self.out_dim, Ws, bs, bns, capi.ptr(self.blob), nbytes,
                                                   capi.stream()))
        self._ws, self._ws_key = None, None

    def __call__(self, img01_nhwc: torch.Tensor, out: torch.Tensor = None) -> torch.Tensor:
        """[B,H,W,3] fp32 in [0,1] (NOT yet 2x-1) -> [B,H/8,W/8,out_dim] fp32."""
        capi, lib = self.capi, self.capi.lib
        B, H, W, _ = img01_nhwc.shape
        x = img01_nhwc.contiguous().float()
        with torch.cuda.device(self.device):
            if self._ws_key != (B, H, W):
                self._ws_bytes = capi.size_query(lib.rb_encoder_workspace_bytes, self.small, B, H, W)
                self._ws = torch.zeros(self._ws_bytes, dtype=torch.uint8, device=self.device)
                self._ws_key = (B, H, W)
            if out is None:
                out = torch.empty(B, -(-H // 8), -(-W // 8), self.out_dim, dtype=torch.float32, device=self.device)
            capi.check(lib.rb_encoder_forward(self.small, self.norm, capi.ptr(self.blob), capi.ptr(x), capi.ptr(out), B, H, W,
                                              self.out_dim, capi.ptr(self._ws), self._ws_bytes, capi.stream()))
        return out
