"""TEST INFRASTRUCTURE ONLY -- never imported by the product (deblurgs_b200/).

Torch restatement of the projection with the antialiasing option (Mip-Splatting's screen-space filter, DESIGN.md
section 3): the opacity a Gaussian blends with is opacity * rho, rho = sqrt(max(det0 / det, 2.5e-5)), det0 and det
the determinants of the projected 2-D covariance before and after its 0.3 px^2 dilation.  Everything else (conic,
radius, tile rectangle, depth, colour) is raster_torch_cpu.project's, operation for operation, and the tile lists and
the composite are raster_torch_cpu's own, so with rho forced to 1 this module reproduces raster_torch_cpu exactly.
Unlike raster_torch_cpu.project it also takes precomputed colours and precomputed 3-D covariances.

Run it in float64 where it serves as truth; its autograd is the gradient oracle of the antialiased backward.
"""
import torch

from . import raster_torch_cpu as rt

H_DILATION = 0.3
R_MIN = 2.5e-5


def aa_rho(a0, b, c0, h=H_DILATION):
    """rho of the undilated 2-D covariance (a0, b; b, c0)."""
    det0 = a0 * c0 - b * b
    det = (a0 + h) * (c0 + h) - b * b
    return torch.sqrt(torch.clamp_min(det0 / det, R_MIN))


def cov3d_from_scale_rot(scales, rots):
    """(S R)^T (S R) with the un-normalised quaternion (r, x, y, z), as raster_torch_cpu.project builds it."""
    P = scales.shape[0]
    r, x, y, z = rots.unbind(1)
    R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
                     2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
                     2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], 1).view(P, 3, 3)
    L = R * scales[:, None, :]
    return L @ L.transpose(1, 2)


def cov3d_from_upper(cov6):
    """[P,6] upper triangle (xx, xy, xz, yy, yz, zz) -> [P,3,3]."""
    a, b, c, d, e, f = cov6.unbind(1)
    return torch.stack([a, b, c, b, d, e, c, e, f], 1).view(-1, 3, 3)


def project(means, opac, view, proj, W, H, tanx, tany, scales=None, rots=None, cov3D=None, shs=None, deg=0,
            campos=None, colors=None, antialiasing=False):
    """raster_torch_cpu.project with precomputed-input options and `antialiasing`.  Adds `rho` and the undilated
    2-D covariance `cov2d0` = (a0, b, c0) to the returned dict."""
    P = means.shape[0]
    hom = torch.cat([means, torch.ones_like(means[:, :1])], 1)
    pv = hom @ view
    ph = hom @ proj
    pw = 1.0 / (ph[:, 3] + 1e-7)
    ndc = ph[:, :2] * pw[:, None]
    Sigma = cov3d_from_upper(cov3D) if cov3D is not None else cov3d_from_scale_rot(scales, rots)
    fx, fy = W / (2 * tanx), H / (2 * tany)
    tz = pv[:, 2]
    limx, limy = 1.3 * tanx, 1.3 * tany
    tx = torch.clamp(pv[:, 0] / tz, -limx, limx) * tz
    ty = torch.clamp(pv[:, 1] / tz, -limy, limy) * tz
    zero = torch.zeros_like(tz)
    J = torch.stack([fx / tz, zero, -(fx * tx) / (tz * tz), zero, fy / tz, -(fy * ty) / (tz * tz)], 1).view(P, 2, 3)
    T = J @ view[:3, :3].t()[None]
    cov = T @ Sigma @ T.transpose(1, 2)
    a0, b, c0 = cov[:, 0, 0], cov[:, 0, 1], cov[:, 1, 1]
    a, c = a0 + H_DILATION, c0 + H_DILATION
    det = a * c - b * b
    det_inv = 1.0 / det
    conic = torch.stack([c * det_inv, -b * det_inv, a * det_inv], 1)
    mid = 0.5 * (a + c)
    disc = torch.sqrt(torch.clamp_min(mid * mid - det, 0.1))
    radius = torch.ceil(3.0 * torch.sqrt(torch.maximum(mid + disc, mid - disc))).detach()
    px = ((ndc[:, 0] + 1.0) * W - 1.0) * 0.5
    py = ((ndc[:, 1] + 1.0) * H - 1.0) * 0.5
    tiles_x, tiles_y = (W + rt.TILE - 1) // rt.TILE, (H + rt.TILE - 1) // rt.TILE
    with torch.no_grad():
        x0 = ((px - radius) / rt.TILE).to(torch.int64).clamp(0, tiles_x)
        y0 = ((py - radius) / rt.TILE).to(torch.int64).clamp(0, tiles_y)
        x1 = ((px + radius + rt.TILE - 1) / rt.TILE).to(torch.int64).clamp(0, tiles_x)
        y1 = ((py + radius + rt.TILE - 1) / rt.TILE).to(torch.int64).clamp(0, tiles_y)
        vis = (tz > 0.2) & (det != 0) & ((x1 - x0) * (y1 - y0) > 0)
    if colors is not None:
        rgb = colors
    else:
        dirs = means - campos[None]
        dirs = dirs / dirs.norm(dim=1, keepdim=True)
        rgb = rt._sh_color(shs, deg, dirs)
    rho = aa_rho(a0, b, c0) if antialiasing else torch.ones_like(a0)
    op = opac[:, 0] * rho if antialiasing else opac[:, 0]
    return dict(px=px, py=py, depth=tz, conic=conic, opac=op, rgb=rgb, radius=radius, vis=vis,
                rect=(x0, y0, x1, y1), tiles=(tiles_x, tiles_y), rho=rho, cov2d0=(a0, b, c0))


def render_view(means, opac, view, proj, bg, W, H, tanx, tany, antialiasing=False, **inputs):
    """(image [3,H,W], projection dict).  `inputs`: scales + rots or cov3D, shs + deg + campos or colors.
    The tile lists sort on float32 depth bits, as the library does, whatever the working precision."""
    pre = project(means, opac, view, proj, W, H, tanx, tany, antialiasing=antialiasing, **inputs)
    point_list, bounds = rt.bin_tiles(dict(pre, depth=pre["depth"].float()))
    return rt.composite(pre, point_list, bounds, bg, W, H), pre
