"""Alpha compositing of foreground renders over a background, in image space or in BEV.

Mirror of /root/reference/bev/tool/compo.py (same function names, argument order and return
values) on CUDA tensors: the three ``cv2.warpPerspective`` calls of ``composite_bev_img``
(compo.py:38,46,47) and the blend become ONE kernel (``bevk_composite_bev_u8c3``: gather three
windows, interpolate, blend in registers, write the composite once); shapes that kernel does not
take go through batched warps and ``bevk_composite_u8c3``, which is also the float64 numpy blend of
``composite_reg_img`` (compo.py:16-23) on its own.  Results are bit-identical to the reference on
the same inputs.

The reference also accepts file names (``cv2.imread``); file IO is outside the hot path, so only
tensors are taken here: uint8 CUDA tensors of shape (H, W, 3) or batches (N, H, W, 3).
"""
import numpy as np

from . import _native
from .homo import homo_from_KRt, INTER_LINEAR


def _check_inputs(*tensors):
    for t in tensors:
        if isinstance(t, str):
            raise TypeError("bev_b200.compo takes CUDA tensors, not file names (image decoding is "
                            "outside the accelerated path)")


def _to_gray_bgr(fg):
    """cv2.cvtColor(cv2.cvtColor(fg, BGR2GRAY), GRAY2BGR) (compo.py:13-14) on the GPU."""
    import torch
    full = torch.full_like(fg, 255)
    return _native.composite_u8c3(fg, fg, full, bw_mode=True)


def composite_reg_img(bg, fg, fg_mask, bw_mode=False):
    """round(fg * mask/255 + bg * (1 - mask/255)) as uint8 (reference compo.py:5-24)."""
    _check_inputs(bg, fg, fg_mask)
    return _native.composite_u8c3(bg, fg, fg_mask, bw_mode=bw_mode)


def composite_bev_img(bg, fg, fg_mask, H_world2bev, H_img2world_fix, K, RT, x_size, y_size,
                      bw_mode=False):
    """Warp background (fixed camera) and foreground + mask (rendering camera K, RT) to the BEV of
    size (x_size, y_size) and blend them (reference compo.py:26-50).
    Returns (composite, H_world2img_cam) like the reference."""
    import torch
    _check_inputs(bg, fg, fg_mask)
    if bw_mode:
        fg = _to_gray_bgr(fg)
    H_world2bev = np.asarray(H_world2bev, np.float64)
    H_img2bev_fix = H_world2bev.dot(np.asarray(H_img2world_fix, np.float64))
    H_world2img_cam = homo_from_KRt(K, Rt_homo=RT)
    H_img2world_cam = np.linalg.inv(H_world2img_cam)
    H_img2bev_cam = H_world2bev.dot(H_img2world_cam)
    single = bg.dim() == 3
    b4, f4, m4 = (t[None] if single else t for t in (bg, fg, fg_mask))
    dsize = (int(x_size), int(y_size))
    compo = composite_bev_batch(b4, f4, m4, H_img2bev_fix, H_img2bev_cam, dsize)
    return (compo[0] if single else compo), H_world2img_cam


def composite_bev_batch(bg, fg, fg_mask, H_img2bev_bg, H_img2bev_fg, dsize, fused=None):
    """N composites in one call: bg (N or 1, Hb, Wb, 3), fg / fg_mask (N, Hf, Wf, 3), homographies
    3x3 (shared) or (N, 3, 3) (one rendering camera per frame) -> (N, height, width, 3).

    The batched form of compo.py:36-49.  ``fused=None`` picks the one-pass kernel
    (bevk_composite_bev_u8c3) whenever the shapes allow it, else three warps and a blend;
    True / False force one route (both give identical bytes).

    The homographies may also both be CUDA tensors on fg's device (e.g. a rendering camera's pose
    made in torch): the kernels of either route then read them when they run, with no host sync, and
    a captured CUDA graph replays whatever matrices were last written into them."""
    import torch
    n = fg.shape[0]
    dmat = any(isinstance(H, torch.Tensor) and H.is_cuda for H in (H_img2bev_bg, H_img2bev_fg))
    if dmat:
        Hb = _native._composite_mats(H_img2bev_bg, "H_img2bev_bg", fg.device).reshape(-1, 3, 3)
        Hf = _native._composite_mats(H_img2bev_fg, "H_img2bev_fg", fg.device).reshape(-1, 3, 3)
        composite_bev, warp = _native.composite_bev_u8c3_dmat, _native.warp_perspective_dmat
    else:
        Hb = np.asarray(H_img2bev_bg, np.float64).reshape(-1, 3, 3)
        Hf = np.asarray(H_img2bev_fg, np.float64).reshape(-1, 3, 3)
        composite_bev, warp = _native.composite_bev_u8c3, _native.warp_perspective
    can_fuse = _native.composite_bev_fusable(bg, fg, dsize)
    if fused is None:
        fused = can_fuse
    if fused:
        return composite_bev(bg, fg, fg_mask, Hb, Hf, dsize)
    if bg.shape[0] == 1 and len(Hb) > 1:  # one background seen through a camera per frame
        bg = bg.expand(n, -1, -1, -1).contiguous()
    bg_bev = warp(bg, Hb if len(Hb) > 1 else Hb[0], dsize, flags=INTER_LINEAR)
    if bg_bev.shape[0] != n:
        bg_bev = bg_bev.expand(n, -1, -1, -1)
    if len(Hf) == 1:
        fm = warp(torch.cat([fg, fg_mask], 0), Hf[0], dsize, flags=INTER_LINEAR)
    else:  # mat_index stays on the host
        idx = np.concatenate([np.arange(n, dtype=np.int32)] * 2)
        fm = warp(torch.cat([fg, fg_mask], 0), Hf, dsize, flags=INTER_LINEAR, mat_index=idx)
    return _native.composite_u8c3(bg_bev.contiguous(), fm[:n], fm[n:])
