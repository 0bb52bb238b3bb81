"""GPU versions of what the reference does with the disparity map after the hot path:
accuracy metrics (depth_estimation_pipeline_metrics.py:18-56) and the point cloud
(depth_estimation_pipeline_hooks.py:84-92, helpers/point_cloud_helpers.py:5-13); and the left-right check with the
background fill for callers that hold both views' disparity maps; and the rectification remap for callers that want
a rectified image itself (to colour a point cloud or display a map); and cv2.reprojectImageTo3D, the metric point
map of a calibrated rig."""
import ctypes
import math

import numpy as np
import torch

from . import _native as N


def _check(rc, what):
    if rc != N.SD_OK:
        raise RuntimeError(f"{what} failed ({rc})")


def evaluate(disparity_estimate: torch.Tensor, disparity_gt: torch.Tensor, max_disparity: float, threshold: float = 3.0):
    """One fused pass: {'D1', 'Threshold_<n>', 'MAE', 'count'} over the mask 0 < gt <= max_disparity."""
    est = disparity_estimate.contiguous().float()
    gt = disparity_gt.to(est.device).contiguous().float()
    if est.shape != gt.shape or not est.is_cuda:
        raise RuntimeError("disparity_estimate and disparity_gt must be CUDA tensors of the same shape")
    out = torch.empty(4, dtype=torch.float64, device=est.device)
    stream = torch.cuda.current_stream(est.device).cuda_stream
    with torch.cuda.device(est.device):   # the launch must happen on the tensors' device, whatever is current
        _check(N.lib().sd_metrics(est.data_ptr(), gt.data_ptr(), est.numel(), float(max_disparity), float(threshold),
                                  out.data_ptr(), stream), "sd_metrics")
    cnt, d1, th, s = out.tolist()
    if cnt == 0:
        return {"D1": float("nan"), f"Threshold_{int(threshold)}": float("nan"), "MAE": float("nan"), "count": 0}
    return {"D1": d1 / cnt, f"Threshold_{int(threshold)}": th / cnt, "MAE": s / cnt, "count": int(cnt)}


def point_cloud(disparity_map: torch.Tensor, focal_length: float, baseline: float, invalid_disparity: float = -1.0):
    """[P,3] tensor of (column, row, depth) for every valid pixel, row-major like the reference's double loop."""
    d = disparity_map.contiguous().float()
    if d.dim() != 2 or not d.is_cuda:
        raise RuntimeError("disparity_map must be a 2-D CUDA tensor")
    H, W = d.shape
    nb = (H * W + 1023) // 1024
    xyz = torch.empty((H * W, 3), dtype=torch.float32, device=d.device)
    scratch = torch.empty(nb + 1, dtype=torch.int32, device=d.device)
    stream = torch.cuda.current_stream(d.device).cuda_stream
    with torch.cuda.device(d.device):
        _check(N.lib().sd_point_cloud(d.data_ptr(), H, W, float(baseline) * float(focal_length), float(invalid_disparity),
                                      xyz.data_ptr(), scratch.data_ptr(), stream), "sd_point_cloud")
    return xyz[: int(scratch[nb].item())]


def left_right_fill(left_map: torch.Tensor, right_map: torch.Tensor, tolerance: float, invalid_disparity: float = -1.0,
                    out=None):
    """Left-right check plus background fill (StereoMatching.set_left_right_check(..., background_fill=True)) of
    [H,W] or [N,H,W] float32 CUDA maps: `left_map` unchecked, `right_map` the right view's map in right-image columns.
    Returns `out` (a new tensor when None); `out` may be `left_map` (in place), not `right_map`."""
    if not (isinstance(left_map, torch.Tensor) and isinstance(right_map, torch.Tensor)):
        raise TypeError("left_map and right_map must be tensors")
    if (left_map.shape != right_map.shape or left_map.dim() not in (2, 3) or not left_map.is_cuda
            or right_map.device != left_map.device):
        raise RuntimeError("left_map and right_map must be CUDA tensors of the same [H,W] or [N,H,W] shape and device")
    for t, name in ((left_map, "left_map"), (right_map, "right_map")):
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise RuntimeError(f"{name} must be a contiguous float32 tensor")
    if out is None:
        out = torch.empty_like(left_map)
    elif (not isinstance(out, torch.Tensor) or out.shape != left_map.shape or out.dtype != torch.float32
          or out.device != left_map.device or not out.is_contiguous()):
        raise RuntimeError("out must be a contiguous float32 tensor of the maps' shape and device")
    if out.data_ptr() == right_map.data_ptr():
        raise RuntimeError("out must not be right_map")
    tolerance = float(tolerance)
    if not math.isfinite(tolerance) or tolerance < 0:
        raise ValueError(f"tolerance must be finite and >= 0, got {tolerance}")
    n = 1 if left_map.dim() == 2 else left_map.shape[0]
    H, W = left_map.shape[-2:]
    if n == 0 or H == 0 or W == 0:
        return out
    stream = torch.cuda.current_stream(left_map.device).cuda_stream
    with torch.cuda.device(left_map.device):
        _check(N.lib().sd_lr_fill(left_map.data_ptr(), right_map.data_ptr(), n, H, W, tolerance,
                                  float(invalid_disparity), out.data_ptr(), stream), "sd_lr_fill")
    return out


def rectify(images: torch.Tensor, map_x: torch.Tensor, map_y: torch.Tensor, out=None):
    """cv2.remap(image, map_x, map_y, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0) of every [H,W]
    plane of a [..., H, W] uint8 or float32 CUDA tensor (e.g. [3,H,W] CHW or [N,3,H,W]), bit for bit (DESIGN.md §14).
    map_x / map_y: float32 [H,W] (cv2.initUndistortRectifyMap with m1type=cv2.CV_32FC1), on the images' device.
    Returns `out` (a new tensor when None), which must not be `images`."""
    if not all(isinstance(t, torch.Tensor) for t in (images, map_x, map_y)):
        raise TypeError("images, map_x and map_y must be tensors")
    if images.dim() < 2 or not images.is_cuda or images.dtype not in (torch.uint8, torch.float32):
        raise RuntimeError("images must be a uint8 or float32 CUDA tensor of shape [..., H, W]")
    H, W = images.shape[-2:]
    for t, name in ((map_x, "map_x"), (map_y, "map_y")):
        if t.dtype != torch.float32 or tuple(t.shape) != (H, W) or t.device != images.device:
            raise RuntimeError(f"{name} must be a float32 [{H},{W}] map (m1type=cv2.CV_32FC1) on {images.device}")
    images, map_x, map_y = images.contiguous(), map_x.contiguous(), map_y.contiguous()
    if out is None:
        out = torch.empty_like(images)
    elif (not isinstance(out, torch.Tensor) or out.shape != images.shape or out.dtype != images.dtype
          or out.device != images.device or not out.is_contiguous()):
        raise RuntimeError("out must be a contiguous tensor of the images' shape, dtype and device")
    if out.data_ptr() == images.data_ptr():
        raise RuntimeError("out must not be images: the remap gathers, it cannot run in place")
    planes = images.numel() // max(1, H * W)
    if planes == 0:
        return out
    stream = torch.cuda.current_stream(images.device).cuda_stream
    with torch.cuda.device(images.device):
        _check(N.lib().sd_rectify(map_x.data_ptr(), map_y.data_ptr(), images.data_ptr(), out.data_ptr(),
                                  N.SD_U8 if images.dtype == torch.uint8 else N.SD_F32, planes, H, W, stream),
               "sd_rectify")
    return out


def reprojection_matrix(Q) -> np.ndarray:
    """Q (cv2.stereoRectify's 4x4 reprojection matrix: numpy array, tensor or nested lists of any integer or float
    dtype) as a contiguous float64 numpy array, the conversion cv2.reprojectImageTo3D makes (it refuses bool)."""
    if isinstance(Q, torch.Tensor):
        Q = Q.detach().cpu().numpy()
    q = np.asarray(Q)
    if q.shape != (4, 4) or q.dtype.kind not in "iuf":
        raise RuntimeError(f"Q must be a 4x4 integer or floating-point matrix (cv2.stereoRectify's Q), got {q.dtype} "
                           f"{q.shape}")
    return np.ascontiguousarray(q, dtype=np.float64)


def reproject_image_to_3d(disparity: torch.Tensor, Q, handle_missing_values: bool = False, out=None):
    """cv2.reprojectImageTo3D(disparity, Q, handleMissingValues=handle_missing_values) of a [H,W] or [N,H,W] float32
    CUDA disparity map, bit for bit (DESIGN.md §15): [..., H, W, 3] float32 points (X, Y, Z).  Q: 4x4 of any integer or
    float dtype, converted to float64 as OpenCV does.  With handle_missing_values, pixels within FLT_EPSILON of their
    frame's minimum disparity get Z = 10000; the minimum is over the non-NaN values (OpenCV's is undefined with NaN).
    Returns `out` (a new tensor when None), which must not overlap `disparity`."""
    if not isinstance(disparity, torch.Tensor):
        raise TypeError("disparity must be a tensor")
    if disparity.dim() not in (2, 3) or not disparity.is_cuda or disparity.dtype != torch.float32:
        raise RuntimeError("disparity must be a float32 CUDA tensor of shape [H,W] or [N,H,W]")
    q = reprojection_matrix(Q)
    disparity = disparity.contiguous()
    shape = tuple(disparity.shape) + (3,)
    if out is None:
        out = torch.empty(shape, dtype=torch.float32, device=disparity.device)
    elif (not isinstance(out, torch.Tensor) or tuple(out.shape) != shape or out.dtype != torch.float32
          or out.device != disparity.device or not out.is_contiguous()):
        raise RuntimeError(f"out must be a contiguous float32 tensor of shape {list(shape)} on {disparity.device}")
    if disparity.numel() == 0:
        return out
    d0, x0 = disparity.data_ptr(), out.data_ptr()
    if x0 < d0 + 4 * disparity.numel() and d0 < x0 + 4 * out.numel():
        raise RuntimeError("out must not overlap disparity")
    n = 1 if disparity.dim() == 2 else disparity.shape[0]
    H, W = disparity.shape[-2:]
    stream = torch.cuda.current_stream(disparity.device).cuda_stream
    with torch.cuda.device(disparity.device):
        _check(N.lib().sd_reproject(d0, n, H, W, q.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                    1 if handle_missing_values else 0, x0, stream), "sd_reproject")
    return out
