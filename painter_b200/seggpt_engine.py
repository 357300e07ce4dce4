"""B200-side mirror of SegGPT/SegGPT_inference/seggpt_engine.py (SURVEY §8 f.2): the same three entry points

    run_one_image(img, tgt, model, device)                                   seggpt_engine.py:26-53
    inference_image(model, device, img_path, img2_paths, tgt2_paths, out_path)       :56-103
    inference_video(model, device, vid_path, num_frames, img2_paths, tgt2_paths, out_path)  :106-181

with identical arguments and results, but with everything between the decoded uint8 pixels and the finished uint8
frame on the GPU: stitch + ImageNet normalisation + nhwc->nchw (pk_stitch_normalize), the forward (one CUDA-graph
replay, painter_b200/graphs.py), unpatchify + bottom half + de-normalisation + clip (pk_seg_postprocess), nearest
resize to the source size + alpha blend (pk_nearest_blend).  Image / video decoding, PIL resizing to 448x448 and file
output stay on the host (file I/O is out of scope, SURVEY §2 row 5); the video path keeps its rolling prompt cache
(previous frames and their binarised predictions, seggpt_engine.py:13-23,128-171) resident in HBM, so a frame costs
one 0.6 MB upload however many cached prompts vote on it.
"""
import ctypes

import numpy as np
import torch

from . import ops
from ._lib import check, lib
from .graphs import GraphedForward

imagenet_mean = np.array([0.485, 0.456, 0.406])
imagenet_std = np.array([0.229, 0.224, 0.225])

_DT = {torch.uint8: 0, torch.float32: 1, torch.float64: 2}


class Cache(list):
    """seggpt_engine.py:13-23: bounded FIFO of prompt frames."""

    def __init__(self, max_size=0):
        super().__init__()
        self.max_size = max_size

    def append(self, x):
        if self.max_size <= 0:
            return
        super().append(x)
        if len(self) > self.max_size:
            self.pop(0)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _graphed(model):
    g = model.__dict__.get("_pk_graphed")
    if g is None:
        g = GraphedForward(model)
        model.__dict__["_pk_graphed"] = g
    return g


def stitch_normalize(tops, bottoms, S):
    """tops / bottoms: lists of P device tensors [S, S, 3] (uint8, or fp32 / fp64 in [0, 1]) -> fp32 [P, 3, 2S, S]."""
    P = len(tops)
    assert P == len(bottoms) and 1 <= P <= 16
    dev = tops[0].device
    for t in list(tops) + list(bottoms):
        assert t.is_cuda and t.is_contiguous() and tuple(t.shape) == (S, S, 3) and t.dtype in _DT, (t.shape, t.dtype)
    arr = ctypes.c_void_p * P
    ia = ctypes.c_int * P
    out = torch.empty((P, 3, 2 * S, S), dtype=torch.float32, device=dev)
    check(lib().pk_stitch_normalize(arr(*[t.data_ptr() for t in tops]), ia(*[_DT[t.dtype] for t in tops]),
                                    arr(*[t.data_ptr() for t in bottoms]), ia(*[_DT[t.dtype] for t in bottoms]),
                                    ctypes.c_void_p(out.data_ptr()), P, S, _stream()), "pk_stitch_normalize")
    return out


def seg_postprocess(patch, h, w, p, want_bin=False):
    """patchified prediction [B, h*w, p*p*3] fp32 -> (fp64 [h*p/2, w*p, 3] in [0, 255], optional fp32 {0,1} mask)."""
    assert patch.dtype == torch.float32 and patch.is_contiguous()
    out = torch.empty((h * p // 2, w * p, 3), dtype=torch.float64, device=patch.device)
    b = torch.empty((h * p // 2, w * p), dtype=torch.float32, device=patch.device) if want_bin else None
    check(lib().pk_seg_postprocess(ctypes.c_void_p(patch.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                   ctypes.c_void_p(b.data_ptr()) if b is not None else None, h, w, p, _stream()),
          "pk_seg_postprocess")
    return out, b


def nearest_blend(seg, image_u8):
    """seg fp64 [SH, SW, 3] (0..255), image uint8 [OH, OW, 3] (device) -> uint8 [OH, OW, 3] blended overlay."""
    OH, OW, _ = image_u8.shape
    dst = torch.empty_like(image_u8)
    check(lib().pk_nearest_blend(ctypes.c_void_p(seg.data_ptr()), seg.shape[0], seg.shape[1],
                                 ctypes.c_void_p(image_u8.data_ptr()), ctypes.c_void_p(dst.data_ptr()), OH, OW,
                                 _stream()), "pk_nearest_blend")
    return dst


def _half_mask(model, device):
    n = model.patch_embed.num_patches
    m = torch.zeros(1, n, device=device)
    m[:, n // 2:] = 1
    return m


def _forward(model, x, tgt, device):
    """The call of seggpt_engine.py:36-47 on device tensors x, tgt [P, 3, 896, 448] fp32; returns patchify(pred)."""
    P = x.shape[0]
    key = ("seg_consts", P, str(device), model.seg_type)
    c = model.__dict__.get("_pk_seg_consts")
    if c is None or c[0] != key:
        seg_type = torch.ones([P, 1], device=device) if model.seg_type == 'instance' else \
            torch.zeros([P, 1], device=device)
        c = (key, _half_mask(model, device), torch.ones((P, 3, x.shape[2], x.shape[3]), device=device), seg_type)
        model.__dict__["_pk_seg_consts"] = c
    _, mask, valid, seg_type = c
    feat_ensemble = 0 if P > 1 else -1
    _, y, _ = _graphed(model)(x, tgt, mask, valid, seg_type, feat_ensemble)
    return y


@torch.no_grad()
def run_one_image(img, tgt, model, device):
    """img, tgt: numpy [P, 896, 448, 3] (already ImageNet-normalised, float64 as the reference callers build them).
    Returns what the reference returns: a CPU float64 tensor [448, 448, 3], the de-normalised bottom half in [0, 255]."""
    device = torch.device(device)
    x = torch.as_tensor(img)
    t = torch.as_tensor(tgt)
    P, H, W, _ = x.shape
    # pk_nhwc_to_nchw_f32 reads packed NHWC: .to() keeps a strided (e.g. permuted) array's strides, so pack it
    xd, td = x.to(device, non_blocking=True).contiguous(), t.to(device, non_blocking=True).contiguous()
    xin = torch.empty((P, 3, H, W), dtype=torch.float32, device=device)
    tin = torch.empty((P, 3, H, W), dtype=torch.float32, device=device)
    for src, dst in ((xd, xin), (td, tin)):
        assert src.dtype in (torch.float32, torch.float64)
        check(lib().pk_nhwc_to_nchw_f32(ctypes.c_void_p(src.data_ptr()), int(src.dtype == torch.float64),
                                        ctypes.c_void_p(dst.data_ptr()), P, H, W, _stream()), "pk_nhwc_to_nchw_f32")
    y = _forward(model, xin, tin, device)
    p = model.patch_size
    out, _ = seg_postprocess(y, H // p, W // p, p)
    return out.cpu()


def _load_prompt(img2_path, tgt2_path, res, hres, device):
    from PIL import Image
    img2 = Image.open(img2_path).convert("RGB").resize((res, hres))
    tgt2 = Image.open(tgt2_path).convert("RGB").resize((res, hres), Image.NEAREST)
    return (torch.from_numpy(np.array(img2)).to(device), torch.from_numpy(np.array(tgt2)).to(device))


@torch.no_grad()
def segment(model, device, image_u8, prompts, want_bin=False):
    """image_u8: device uint8 [448, 448, 3] (the query, resized); prompts: list of (prompt image, prompt target)
    device tensors [448, 448, 3] (uint8, or float in [0,1] for cached video frames).  Returns (fp64 [448, 448, 3] in
    [0, 255], optional binarised mask) - seggpt_engine.py:65-93 without the host arithmetic."""
    S = image_u8.shape[0]
    x = stitch_normalize([p[0] for p in prompts], [image_u8] * len(prompts), S)
    t = stitch_normalize([p[1] for p in prompts], [p[1] for p in prompts], S)      # "tgt is not available"
    torch.manual_seed(2)      # seggpt_engine.py:91 (no random op follows in eval mode; kept for RNG-state parity)
    y = _forward(model, x, t, device)
    p = model.patch_size
    return seg_postprocess(y, 2 * S // p, S // p, p, want_bin=want_bin)


def inference_image(model, device, img_path, img2_paths, tgt2_paths, out_path):
    from PIL import Image
    device = torch.device(device)
    res, hres = 448, 448
    image = Image.open(img_path).convert("RGB")
    input_image = torch.from_numpy(np.array(image)).to(device)
    image_r = torch.from_numpy(np.array(image.resize((res, hres)))).to(device)
    prompts = [_load_prompt(a, b, res, hres, device) for a, b in zip(img2_paths, tgt2_paths)]
    out, _ = segment(model, device, image_r, prompts)
    blended = nearest_blend(out, input_image)
    Image.fromarray(blended.cpu().numpy()).save(out_path)
    return blended


def inference_video(model, device, vid_path, num_frames, img2_paths, tgt2_paths, out_path):
    import cv2
    from PIL import Image
    device = torch.device(device)
    res, hres = 448, 448
    cap = cv2.VideoCapture(vid_path)
    fps = cap.get(cv2.CAP_PROP_FPS)
    width = int(cap.get(cv2.CAP_PROP_FRAME_WIDTH))
    height = int(cap.get(cv2.CAP_PROP_FRAME_HEIGHT))
    fourcc = cv2.VideoWriter_fourcc(*'mp4v')
    video_writer = cv2.VideoWriter(out_path, fourcc, fps, (width, height), True)
    if img2_paths is None:
        _, frame = cap.read()
        img2 = Image.fromarray(frame[:, :, ::-1]).convert('RGB')
    else:
        img2 = Image.open(img2_paths[0]).convert("RGB")
    img2 = torch.from_numpy(np.array(img2.resize((res, hres)))).to(device)
    tgt2 = Image.open(tgt2_paths[0]).convert("RGB").resize((res, hres), Image.NEAREST)
    tgt2 = torch.from_numpy(np.array(tgt2)).to(device)
    frames_cache, target_cache = Cache(num_frames), Cache(num_frames)
    n = 0
    while True:
        ret, frame = cap.read()
        if not ret:
            break
        image = Image.fromarray(frame[:, :, ::-1]).convert('RGB')
        input_image = torch.from_numpy(np.array(image)).to(device)
        image_r = torch.from_numpy(np.array(image.resize((res, hres)))).to(device)
        prompts = list(zip([img2] + frames_cache, [tgt2] + target_cache))
        out, binm = segment(model, device, image_r, prompts, want_bin=num_frames > 0)
        frames_cache.append(image_r)
        if num_frames > 0:
            target_cache.append(binm.unsqueeze(-1).expand(-1, -1, 3).contiguous())
        blended = nearest_blend(out, input_image)
        video_writer.write(np.ascontiguousarray(blended.cpu().numpy()[:, :, ::-1]))
        n += 1
    video_writer.release()
    return n
