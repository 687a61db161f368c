"""fp64 reference of the forward-backward consistency check (F5, rb_flow_consistency) for the tests: a plain torch-CPU
restatement of the test the kernel implements, kept beside the tests that compare against it.  The check is an extension:
the reference project has no counterpart, so this is not part of oracle/raft_oracle.py (which restates the reference)."""
import torch

Tensor = torch.Tensor


def fb_consistency(flow_fw: Tensor, flow_bw: Tensor, scale: float = 1.0, alpha1: float = 0.01,
                   alpha2: float = 0.5, return_margin: bool = False):
    """Occlusion codes of both directions, [B,H,W] uint8 each, for flows [B,H,W,2] (x, y), in fp64.
    At pixel p with u = scale*f(p) and t = p + u: 2 if t lies outside [0,W-1] x [0,H-1], else with
    g' = scale*bilinear(g, t) (corners floor(t), min(floor(t)+1, dim-1)) 1 if |u + g'|^2 >= alpha1 (|u|^2 + |g'|^2)
    + alpha2, else 0 (Sundaram et al. 2010; UnFlow, Meister et al. 2018).  Inside the frame the bilinear sample equals
    the reference's truncating sampler (networks/utils.py:40-99) in real arithmetic.  With return_margin, also per
    direction (lhs - rhs, rhs, distance of t to the nearest frame border; signed, negative outside) for tie analysis."""
    def one(f, g):
        B, H, W, _ = f.shape
        f, g = f.double(), g.double()
        ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float64), torch.arange(W, dtype=torch.float64), indexing="ij")
        u = scale * f
        tx, ty = xs + u[..., 0], ys + u[..., 1]
        border = torch.minimum(torch.minimum(tx, (W - 1) - tx), torch.minimum(ty, (H - 1) - ty))
        inside = border >= 0
        cx, cy = tx.clamp(0, W - 1), ty.clamp(0, H - 1)  # only the inside values are used
        x0, y0 = cx.floor(), cy.floor()
        ax, ay = (cx - x0)[..., None], (cy - y0)[..., None]
        x0, y0 = x0.long(), y0.long()
        x1, y1 = (x0 + 1).clamp(max=W - 1), (y0 + 1).clamp(max=H - 1)
        bi = torch.arange(B)[:, None, None]
        gs = ((1 - ax) * (1 - ay) * g[bi, y0, x0] + ax * (1 - ay) * g[bi, y0, x1]
              + (1 - ax) * ay * g[bi, y1, x0] + ax * ay * g[bi, y1, x1]) * scale
        lhs = ((u + gs) ** 2).sum(-1)
        rhs = alpha1 * ((u ** 2).sum(-1) + (gs ** 2).sum(-1)) + alpha2
        occ = torch.where(inside, (lhs >= rhs).to(torch.uint8), torch.full_like(lhs, 2, dtype=torch.uint8))
        return occ, (lhs - rhs, rhs, border)
    (occ_fw, m_fw), (occ_bw, m_bw) = one(flow_fw, flow_bw), one(flow_bw, flow_fw)
    if return_margin:
        return occ_fw, occ_bw, m_fw, m_bw
    return occ_fw, occ_bw
