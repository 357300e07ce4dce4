"""B200-side mirror of the Painter task-inference `run_one_image` functions (SURVEY §8 f.2), e.g.
Painter/eval/ade20k_semantic/painter_inference_segm.py:67-93: same arguments, same PNG on disk, with the
nhwc->nchw conversion, the forward (CUDA-graph replay), unpatchify + bottom half + de-normalisation + clip and the
bilinear resize to the source size on the GPU; only the final uint8 image crosses back to the host."""
import ctypes

import numpy as np
import torch

from ._lib import check, lib
from .seggpt_engine import _graphed, _stream, seg_postprocess


def bilinear_u8(seg, OH, OW):
    """seg fp64 [SH, SW, 3] -> uint8 [OH, OW, 3] = uint8(int(F.interpolate(seg, mode='bilinear')))."""
    dst = torch.empty((OH, OW, 3), dtype=torch.uint8, device=seg.device)
    check(lib().pk_bilinear_u8(ctypes.c_void_p(seg.data_ptr()), seg.shape[0], seg.shape[1],
                               ctypes.c_void_p(dst.data_ptr()), OH, OW, _stream()), "pk_bilinear_u8")
    return dst


@torch.no_grad()
def run_one_image(img, tgt, size, model, out_path, device):
    """img, tgt: numpy [2*S, S, 3] ImageNet-normalised canvases; size = (width, height) of the source image; model: the
    painter_b200 Painter module or a DistributedDataParallel wrapper of it (the script passes `model.module` users)."""
    from PIL import Image
    device = torch.device(device)
    net = model.module if hasattr(model, "module") else model
    # pk_nhwc_to_nchw_f32 reads packed NHWC: .to() keeps a strided (e.g. permuted) array's strides, so pack it
    x = torch.as_tensor(img).unsqueeze(0).to(device, non_blocking=True).contiguous()
    t = torch.as_tensor(tgt).unsqueeze(0).to(device, non_blocking=True).contiguous()
    _, H, W, _ = x.shape
    xin = torch.empty((1, 3, H, W), dtype=torch.float32, device=device)
    tin = torch.empty((1, 3, H, W), dtype=torch.float32, device=device)
    for src, dst in ((x, xin), (t, tin)):
        check(lib().pk_nhwc_to_nchw_f32(ctypes.c_void_p(src.data_ptr()), int(src.dtype == torch.float64),
                                        ctypes.c_void_p(dst.data_ptr()), 1, H, W, _stream()), "pk_nhwc_to_nchw_f32")
    p = net.patch_size
    n = (H // p) * (W // p)
    mask = torch.zeros(1, n, device=device)
    mask[:, n // 2:] = 1
    valid = torch.ones_like(tin)
    _, y, _ = _graphed(net)(xin, tin, mask, valid)
    seg, _ = seg_postprocess(y, H // p, W // p, p)
    out = bilinear_u8(seg, size[1], size[0])
    Image.fromarray(out.cpu().numpy()).save(out_path)
    return out
