#!/usr/bin/env python
"""Drop-in for the reference's ``infer_raft.py`` (same flags and defaults, infer_raft.py:51-67) on the
raft_b200 CUDA engine -- no TensorFlow, no tensorpack.

    python infer_raft.py --im1 frame_0016.png --im2 frame_0017.png --load release_weight/raft-things.npz [--small]

Like the reference it decodes BGR with OpenCV, resizes both frames to 432x1024 (bilinear cv2.resize,
dataflow/test_dataflow.py:85-87), scales to [0,1], runs 20 iterations and writes the colour-coded flow
to ``raft_flow_raft-things.png`` in the working directory (regardless of --small, infer_raft.py:44).
Flags the reference parses but ignores (--gpu, --data, --out, -o) are accepted; ``--batch`` stays 1.
Extensions: --iters, --keep-size (replicate-pad to a multiple of 8 instead of resizing), --npy, --flo, --bidirectional
(also the backward flow, ``raft_flow_backward.png``, and the forward occlusion mask, ``raft_occlusion.png``: consistent
pixels black, occluded white, leaving the frame grey; with --npy X.npy also X_backward.npy and X_occ.npy = [2,H,W] uint8,
forward mask first).
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

OCC_GRAY = np.array([0, 255, 128], dtype=np.uint8)  # occlusion code (consistent, occluded, leaves the frame) -> grey level


def read_pair(im1, im2, size):
    import cv2
    out = []
    for path in (im1, im2):
        with open(path, "rb") as f:
            img = cv2.imdecode(np.asarray(bytearray(f.read()), dtype="uint8"), cv2.IMREAD_COLOR)  # BGR
        if img is None:
            raise FileNotFoundError(path)
        if size is not None:
            img = cv2.resize(img, dsize=(size[1], size[0]))
        out.append(np.float32(img) / 255.0)
    return out[0][None], out[1][None]


def main(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument('--gpu', default='1', help='comma separated list of GPU(s) to use (ignored, as in the reference)')
    p.add_argument('--data', default='', help='unused (reference flag)')
    p.add_argument('--load', default='release_weight/raft-things.npz', help='npz checkpoint keyed by TF variable names')
    p.add_argument('-m', '--mode', default='test', choices=['train', 'val', 'test', 'export', 'flops'])
    p.add_argument('--out', default='./log')
    p.add_argument('--batch', default=1, type=int)
    p.add_argument('-o', '--optimizer', default='adam', choices=['adam', 'adamw', 'sgd', 'sgd_cyclic', 'sgd_1cycle'])
    p.add_argument('--im1', default='frame_0010.png')
    p.add_argument('--im2', default='frame_0011.png')
    p.add_argument('--small', action='store_true')
    p.add_argument('--iters', type=int, default=20, help='extension: GRU iterations (reference: 20)')
    p.add_argument('--keep-size', action='store_true', help='extension: pad to a multiple of 8 instead of resizing to 432x1024')
    p.add_argument('--npy', default=None, help='extension: also save the raw [H,W,2] flow')
    p.add_argument('--flo', default=None, help='extension: also save the flow as a Middlebury .flo file')
    p.add_argument('--bidirectional', action='store_true',
                   help='extension: also compute the backward flow and the forward-backward occlusion masks')
    args = p.parse_args(argv)
    if args.mode != 'test':
        print(f"mode '{args.mode}' has no implementation in the reference either (infer_raft.py:71-95); nothing to do")
        return 0
    from networks import RAFT
    import cv2
    from flow_utils import flow_to_color, write_flo
    left, right = read_pair(args.im1, args.im2, None if args.keep_size else (432, 1024))
    model = RAFT.RAFT(left.shape[1:], args, iters=args.iters).load(args.load)
    if args.bidirectional:
        flow, flow_bw, occ_fw, occ_bw = (t.cpu().numpy() for t in model.forward_backward(left, right))
    else:
        flow = model.forward(left, right).cpu().numpy()
    print(0, flow.shape)
    cv2.imwrite("raft_flow_raft-things.png", flow_to_color(flow[0], convert_to_bgr=True))
    if args.npy:
        np.save(args.npy, flow[0])
    if args.flo:
        write_flo(args.flo, flow[0])
    if args.bidirectional:
        cv2.imwrite("raft_flow_backward.png", flow_to_color(flow_bw[0], convert_to_bgr=True))
        cv2.imwrite("raft_occlusion.png", OCC_GRAY[occ_fw[0]])
        if args.npy:
            stem = args.npy[:-4] if args.npy.endswith(".npy") else args.npy
            np.save(stem + "_backward.npy", flow_bw[0])
            np.save(stem + "_occ.npy", np.stack([occ_fw[0], occ_bw[0]]))
    return 0


if __name__ == '__main__':
    sys.exit(main())
