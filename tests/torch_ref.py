"""Dense fp64 PyTorch restatement of the splatting math (SURVEY.md Appendix A) used to
validate the C++ oracle independently: forward values and -- through autograd -- the
hand-derived backward (A.5/A.6).  O(P*N) memory: small scenes only.

The non-differentiable selections (tile rect membership, alpha < 1/255 skip, power > 0
skip, T < 1e-4 termination, the 0.99 clamp and the 1.3*tanfov clamp) are treated exactly
as the upstream backward treats them: as constants.
"""
import numpy as np
import torch

ALPHA_MIN = 1.0 / 255.0


def quat_to_R(q):
    r, x, y, z = q.unbind(-1)
    return torch.stack([
        1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
        2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
        2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], -1).reshape(-1, 3, 3)


def render(cam, means3D, scales, rotations, opacities, colors, rects, means2D=None,
           sigma_mult=3.0, dtype=torch.float64, tiled=False, sort_depths=None):
    """cam: dict(W,H,tanfovx,tanfovy,view[16],proj[16],bg[3],scale_modifier).
    rects: [N,4] int tile rects (minx,miny,maxx,maxy) from the oracle (0-area = culled).
    tiled: evaluate tile by tile, each tile over the Gaussians whose rect covers it (same values, far less memory).
    sort_depths: [N] fp32 view depths that set the blend order (e.g. the oracle's `depths`); default: this
    function's own depths rounded to fp32.
    Returns color[C,H,W], depth[H,W], final_T[H,W], n_contrib-equivalent weights."""
    W, H = cam["W"], cam["H"]
    V = torch.tensor(np.asarray(cam["view"], dtype=np.float64).reshape(4, 4), dtype=dtype)   # row-vector convention
    Pm = torch.tensor(np.asarray(cam["proj"], dtype=np.float64).reshape(4, 4), dtype=dtype)
    bg = torch.tensor(cam["bg"], dtype=dtype)
    N = means3D.shape[0]
    ones = torch.ones(N, 1, dtype=dtype)
    p4 = torch.cat([means3D, ones], 1)
    t = p4 @ V          # [N,4] (row-vector convention: p_view = p * V)
    hom = p4 @ Pm
    pw = 1.0 / (hom[:, 3] + 1e-7)
    ndc = hom[:, :2] * pw[:, None]
    if means2D is not None:
        ndc = ndc + means2D[:, :2]
    px = ((ndc[:, 0] + 1.0) * W - 1.0) * 0.5
    py = ((ndc[:, 1] + 1.0) * H - 1.0) * 0.5

    R = quat_to_R(rotations)
    s = scales * cam["scale_modifier"]
    Sigma = R @ torch.diag_embed(s * s) @ R.transpose(1, 2)

    fx = W / (2.0 * cam["tanfovx"])
    fy = H / (2.0 * cam["tanfovy"])
    limx, limy = 1.3 * cam["tanfovx"], 1.3 * cam["tanfovy"]
    tx, ty, tz = t[:, 0], t[:, 1], t[:, 2]
    txtz, tytz = (tx / tz).detach(), (ty / tz).detach()
    cx = torch.where((txtz < -limx) | (txtz > limx), (txtz.clamp(-limx, limx) * tz).detach(), tx)
    cy = torch.where((tytz < -limy) | (tytz > limy), (tytz.clamp(-limy, limy) * tz).detach(), ty)
    zero = torch.zeros_like(tz)
    J = torch.stack([fx / tz, zero, -fx * cx / (tz * tz),
                     zero, fy / tz, -fy * cy / (tz * tz)], -1).reshape(N, 2, 3)
    Wr = V[:3, :3].t()   # t = Wr p + tr
    M = J @ Wr
    cov = M @ Sigma @ M.transpose(1, 2)
    a = cov[:, 0, 0] + 0.3
    b = cov[:, 0, 1]
    c = cov[:, 1, 1] + 0.3
    det = a * c - b * b
    cA, cB, cC = c / det, -b / det, a / det

    rects = torch.as_tensor(np.asarray(rects), dtype=torch.long)
    valid = ((rects[:, 2] - rects[:, 0]) * (rects[:, 3] - rects[:, 1]) > 0)

    key = tz.detach().numpy().astype(np.float32) if sort_depths is None else np.asarray(sort_depths, np.float32)
    order = np.lexsort((np.arange(N), key.view(np.uint32)))
    o = torch.as_tensor(order, dtype=torch.long)
    bg_c = torch.cat([bg, torch.zeros(colors.shape[1] - 3, dtype=dtype)]) if colors.shape[1] >= 3 else None
    blend = lambda xs, ys, sel, in_rect: _blend(xs.to(dtype), ys.to(dtype), px[sel], py[sel], cA[sel], cB[sel], cC[sel],
                                                opacities[sel], colors[sel], tz[sel], in_rect, bg_c)

    if not tiled:
        ys, xs = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
        xs, ys = xs.reshape(-1), ys.reshape(-1)
        tile_x, tile_y = xs // 16, ys // 16
        in_rect = (valid[o][None, :]
                   & (tile_x[:, None] >= rects[o, 0][None, :]) & (tile_x[:, None] < rects[o, 2][None, :])
                   & (tile_y[:, None] >= rects[o, 1][None, :]) & (tile_y[:, None] < rects[o, 3][None, :]))
        color, depth, final_T, n_contrib = blend(xs, ys, o, in_rect)
    else:
        # the same blend per 16x16 tile over the tile's own list (the Gaussians whose rect covers it, in the same order):
        # O(pixels x splats per tile) instead of O(pixels x N)
        parts, pix = [], []
        for ty in range((H + 15) // 16):
            for tx in range((W + 15) // 16):
                ys, xs = torch.meshgrid(torch.arange(ty * 16, min(ty * 16 + 16, H)), torch.arange(tx * 16, min(tx * 16 + 16, W)),
                                        indexing="ij")
                xs, ys = xs.reshape(-1), ys.reshape(-1)
                covers = valid[o] & (rects[o, 0] <= tx) & (tx < rects[o, 2]) & (rects[o, 1] <= ty) & (ty < rects[o, 3])
                sel = o[covers]
                parts.append(blend(xs, ys, sel, torch.ones(xs.shape[0], sel.shape[0], dtype=torch.bool)))
                pix.append(ys * W + xs)
        inv = torch.argsort(torch.cat(pix))
        color, depth, final_T, n_contrib = (torch.cat([pt[i] for pt in parts])[inv] for i in range(4))
    return {
        "color": color.t().reshape(-1, H, W), "depth": depth.reshape(H, W),
        "final_T": final_T.reshape(H, W), "n_contrib": n_contrib.reshape(H, W),
        "means2D": torch.stack([px, py], -1), "conic": torch.stack([cA, cB, cC], -1),
        "cov2D": torch.stack([a, b, c], -1), "depths": tz,
    }


def _blend(pxs, pys, px, py, cA, cB, cC, opacities, colors, tz, in_rect, bg):
    """Front-to-back blend of the splats px.. (already in blend order) at the pixels (pxs, pys); in_rect[pixel, splat]
    says which splats are on the pixel's tile list.  -> color[npx,C], depth[npx], final_T[npx], n_contrib[npx]."""
    dx = px[None, :] - pxs[:, None]
    dy = py[None, :] - pys[:, None]
    power = -0.5 * (cA[None, :] * dx * dx + cC[None, :] * dy * dy) - cB[None, :] * dx * dy
    G = torch.exp(power.clamp(max=0.0))
    raw = opacities[None, :] * G
    alpha = raw - (raw - 0.99).clamp(min=0).detach()
    skip = (~in_rect) | (power.detach() > 0) | (alpha.detach() < ALPHA_MIN)
    alpha_eff = torch.where(skip, torch.zeros_like(alpha), alpha)
    one_minus = 1.0 - alpha_eff
    T_after = torch.cumprod(one_minus, dim=1)
    T_before = torch.cat([torch.ones(T_after.shape[0], 1, dtype=T_after.dtype), T_after], 1)[:, :-1]
    stop = (~skip) & (T_after.detach() < 1e-4)
    done = torch.cummax(stop.to(torch.int8), dim=1)[0].bool()
    wgt = torch.where(done, torch.zeros_like(alpha_eff), alpha_eff * T_before)
    applied = (~skip) & (~done)
    # final T = product over applied entries
    final_T = torch.prod(torch.where(applied, one_minus, torch.ones_like(one_minus)), dim=1)
    color = wgt @ colors
    if bg is not None:
        color = color + final_T[:, None] * bg[None, :]
    depth = wgt @ tz
    # position among in-rect entries (the tile list position)
    pos_in_list = torch.cumsum(in_rect.to(torch.long), dim=1)
    n_contrib = torch.where(applied, pos_in_list, torch.zeros_like(pos_in_list)).max(dim=1)[0] \
        if pos_in_list.shape[1] > 0 else torch.zeros(pos_in_list.shape[0], dtype=torch.long)
    return color, depth, final_T, n_contrib
