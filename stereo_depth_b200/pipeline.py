"""Thin shim of the reference's pipeline layer around the "cuda" backend (SURVEY.md section 8-f, rank 1), so the
reference's scripts can run against this backend:

  DepthEstimationPipelineConfig / Result / Context / DepthEstimationPipeline
      <- src/python/pipeline/depth_estimation_pipeline.py:14-87
  extract_config_from_camera, validate_pipeline_config_wrt_camera, run_depth_estimation_pipeline,
  run_depth_estimation_pipeline_evaluation, reduce_metrics
      <- src/python/pipeline/depth_estimation_pipeline_runner.py:12-94
  Camera, EvaluationCamera (the protocol the runner consumes; no dataset readers)
      <- src/python/pipeline/camera/camera.py:7-35
  D1Metric, ThresholdMetric, MAEMetric
      <- src/python/pipeline/depth_estimation_pipeline_metrics.py:18-56 (one fused GPU pass instead of three masked
         tensor expressions: stereo_depth_b200/csrc/consumers.cu)

Right-view synthesis (Deep3D) and the DNN backends are out of scope: `process` needs the right view, or a
user-supplied `right_view_synthesis` object with a `.process(left)` method.
"""
from __future__ import annotations

import time
from abc import ABC, abstractmethod
from contextlib import contextmanager
from dataclasses import dataclass
from typing import Any, Dict, Iterable, Iterator, List, Optional, Tuple

import torch

from . import consumers, cuda_depth
from .backend import CudaStereoMatchingBackend, StereoMatching


@contextmanager
def cuda_perf_clock(label: str, do_log: bool):
    """helpers/torch_helpers.py:19-28: wall time with a device synchronisation, only when logging."""
    if not do_log:
        yield
        return
    torch.cuda.synchronize()
    t0 = time.time()
    yield
    torch.cuda.synchronize()
    print(f"{label}: {(time.time() - t0) * 1000:.3f} ms")


@dataclass
class DepthEstimationPipelineConfig:
    image_shape: Tuple[int, int] = (384, 1280)
    min_disparity: int = 1
    max_disparity: int = 64
    invalid_disparity: float = -1.0
    stereo_matching_backend: str = "cuda"
    log_perf_time: bool = False
    # left-right consistency check tolerance in pixels (None = off); failing pixels get `invalid_disparity`
    left_right_check: Optional[float] = None
    # with left_right_check: fill the pixels it rejects from the background (DESIGN.md §13) instead of marking them
    left_right_background_fill: bool = False
    # raw (unrectified) frames: ((left map_x, left map_y), (right map_x, right map_y)) from cv2.initUndistortRectifyMap
    # with m1type=cv2.CV_32FC1; every frame is rectified on the GPU before matching (None = frames are rectified)
    rectification_maps: Optional[Tuple[Any, Any]] = None
    # the 4x4 reprojection matrix Q of cv2.stereoRectify, in the coordinates of the disparity map (the rectified left
    # view with rectification_maps): every result then carries its metric points (consumers.reproject_image_to_3d)
    reprojection_matrix: Optional[Any] = None

    def update(self, **kwargs: Any) -> "DepthEstimationPipelineConfig":
        for key, value in kwargs.items():
            if not hasattr(self, key):
                raise RuntimeError(f"Unexpected keyword argument: '{key}'.")
            setattr(self, key, value)
        return self


@dataclass
class DepthEstimationResult:
    left_image: torch.Tensor
    right_image: torch.Tensor
    disparity_map: torch.Tensor
    points: Optional[torch.Tensor] = None   # [H,W,3] float32 (X, Y, Z) when config.reprojection_matrix is set


@dataclass
class DepthEstimationPipelineContext:
    disparity_map: torch.Tensor
    left_image: torch.Tensor
    right_image: torch.Tensor
    config: DepthEstimationPipelineConfig
    frame_index: int
    points: Optional[torch.Tensor] = None


class DepthEstimationPipeline:

    def __init__(self, config: Optional[DepthEstimationPipelineConfig] = None, right_view_synthesis=None):
        self._config = config if config is not None else DepthEstimationPipelineConfig()
        self._right_view_synthesis = right_view_synthesis
        self._reprojection = (None if self._config.reprojection_matrix is None
                              else consumers.reprojection_matrix(self._config.reprojection_matrix))
        self._stereo_matching = self._get_stereo_matching()

    def process(self, left_image: torch.Tensor, right_image: Optional[torch.Tensor] = None) -> DepthEstimationResult:
        left_image = left_image.cuda()
        with cuda_perf_clock("Right view generation", self._config.log_perf_time):
            if right_image is None:
                if self._right_view_synthesis is None:
                    raise RuntimeError("right_image is required: right-view synthesis is outside this backend's scope "
                                       "(pass right_view_synthesis= to plug one in)")
                right_image = self._right_view_synthesis.process(left_image)
        with cuda_perf_clock("Stereo matching", self._config.log_perf_time):
            disparity_map = self._stereo_matching.process(left_image, right_image)
        points = None
        if self._reprojection is not None:
            with cuda_perf_clock("Reprojection", self._config.log_perf_time):
                points = consumers.reproject_image_to_3d(disparity_map, self._reprojection)
        return DepthEstimationResult(disparity_map=disparity_map, left_image=left_image, right_image=right_image,
                                     points=points)

    def get_configuration(self) -> DepthEstimationPipelineConfig:
        return self._config

    def _get_stereo_matching(self) -> StereoMatching:
        if self._config.left_right_background_fill and self._config.left_right_check is None:
            raise RuntimeError("left_right_background_fill needs left_right_check (a tolerance in pixels): the fill "
                               "replaces the pixels the check rejects")
        if self._config.stereo_matching_backend == "cuda":
            config = cuda_depth.StereoMatchingConfiguration(
                height=self._config.image_shape[0],
                width=self._config.image_shape[1],
                min_disparity=self._config.min_disparity,
                max_disparity=self._config.max_disparity,
            )
            backend = CudaStereoMatchingBackend(configuration=config)
            if self._config.rectification_maps is not None:
                backend.native.set_rectification(*self._config.rectification_maps)
            if self._config.left_right_check is not None:
                backend.native.set_left_right_check(self._config.left_right_check, self._config.invalid_disparity,
                                                    self._config.left_right_background_fill)
            return backend
        raise RuntimeError(f"Unsupported stereo matching backend: {self._config.stereo_matching_backend}")


class Camera(ABC):
    """camera/camera.py:7-27 -- what the runner needs from an image source."""

    @abstractmethod
    def focal_length(self) -> float:
        pass

    @abstractmethod
    def baseline(self) -> float:
        pass

    @abstractmethod
    def get_image_shape(self) -> Tuple[int, int]:
        pass

    @abstractmethod
    def get_disparity_boundaries(self) -> Tuple[int, int]:
        pass

    @abstractmethod
    def stream_image_pairs(self) -> Iterator[Tuple[torch.Tensor, Optional[torch.Tensor]]]:
        pass


class EvaluationCamera(Camera):
    """camera/camera.py:30-35."""

    @abstractmethod
    def stream_image_pairs_with_gt_disparity(self) -> Iterator[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]]:
        pass


def extract_config_from_camera(camera) -> DepthEstimationPipelineConfig:
    """runner.py:12-19."""
    min_disparity, max_disparity = camera.get_disparity_boundaries()
    return DepthEstimationPipelineConfig(image_shape=camera.get_image_shape(), min_disparity=min_disparity,
                                         max_disparity=max_disparity)


def validate_pipeline_config_wrt_camera(config: DepthEstimationPipelineConfig, camera) -> None:
    """runner.py:22-25 (same comparison, same message)."""
    if camera.get_image_shape() != config.image_shape:
        raise RuntimeError(f"Incompatible image shapes between pipeline configuration and camera."
                           f"Pipeline expects: {config.image_shape} but camera provides: {camera.get_image_shape()}.")


def _is_camera(source) -> bool:
    return hasattr(source, "stream_image_pairs") and hasattr(source, "get_image_shape")


def _check_frame_shape(config, left_view) -> None:
    if tuple(left_view.shape[-2:]) != tuple(config.image_shape):
        raise RuntimeError(f"Incompatible image shapes between pipeline configuration and camera."
                           f"Pipeline expects: {config.image_shape} but camera provides: {tuple(left_view.shape[-2:])}.")


def run_depth_estimation_pipeline(camera, pipeline: DepthEstimationPipeline, hooks: Iterable = None) -> None:
    """Frame loop of runner.py:38-66.  `camera` is anything with the reference's Camera protocol (camera/camera.py:7-27:
    `get_image_shape`, `stream_image_pairs`); a plain iterable of (left, right) pairs is accepted as well.  Hooks are
    objects with on_pipeline_start() / process(context) / on_pipeline_end() (depth_estimation_pipeline_hooks.py:18-32);
    they run in order on the calling thread (the reference's joblib pool is clamped to one job, runner.py:47)."""
    hooks = list(hooks or [])
    config = pipeline.get_configuration()
    if _is_camera(camera):
        validate_pipeline_config_wrt_camera(config, camera)
        image_pairs = camera.stream_image_pairs()
    else:
        image_pairs = camera
    for hook in hooks:
        hook.on_pipeline_start()
    for frame_index, (left_view, right_view) in enumerate(image_pairs):
        _check_frame_shape(config, left_view)
        result = pipeline.process(left_view, right_view)
        context = DepthEstimationPipelineContext(disparity_map=result.disparity_map, left_image=result.left_image,
                                                 right_image=result.right_image, config=config, frame_index=frame_index,
                                                 points=result.points)
        for hook in hooks:
            hook.process(context)
    for hook in hooks:
        hook.on_pipeline_end()


class DepthEstimationPipelineMetric:
    """Interface of depth_estimation_pipeline_metrics.py:7-15.  The built-in metrics are evaluated together by one fused
    kernel over the runner's mask `0 < gt <= max_disparity` (runner.py:85); `process` keeps the reference's signature
    for metrics a user brings along."""

    def name(self) -> str:
        raise NotImplementedError

    def process(self, disparity_estimate: torch.Tensor, disparity_gt: torch.Tensor, mask: torch.Tensor) -> float:
        raise NotImplementedError


class D1Metric(DepthEstimationPipelineMetric):
    def name(self) -> str:
        return "D1"

    def process(self, disparity_estimate, disparity_gt, mask):
        e = torch.abs(disparity_estimate[mask] - disparity_gt[mask])
        return torch.mean(((e > 3) & (e / disparity_gt[mask].abs() > 0.05)).float()).item()


class ThresholdMetric(DepthEstimationPipelineMetric):
    def __init__(self, threshold: float):
        self._threshold = threshold

    def name(self) -> str:
        return f"Threshold_{int(self._threshold)}"

    def process(self, disparity_estimate, disparity_gt, mask):
        e = torch.abs(disparity_estimate[mask] - disparity_gt[mask])
        return torch.mean((e > self._threshold).float()).item()


class MAEMetric(DepthEstimationPipelineMetric):
    def name(self) -> str:
        return "MAE"

    def process(self, disparity_estimate, disparity_gt, mask):
        return torch.nn.functional.l1_loss(disparity_estimate[mask], disparity_gt[mask]).item()


def reduce_metrics(metrics_results: Dict[str, List[float]], reduction: str) -> Dict[str, float]:
    """runner.py:28-35."""
    ops = {"mean": lambda x: sum(x) / len(x), "sum": sum}
    return {key: ops[reduction](value) for key, value in metrics_results.items()}


def run_depth_estimation_pipeline_evaluation(camera, pipeline: DepthEstimationPipeline,
                                             metrics: Iterable[DepthEstimationPipelineMetric] = None,
                                             reduction: str = "mean", verbose: bool = True) -> Dict[str, float]:
    """Evaluation loop of runner.py:69-94.  `camera` follows the reference's EvaluationCamera protocol
    (`stream_image_pairs_with_gt_disparity`, camera/camera.py:30-35) or is a plain iterable of (left, right, gt_disparity).
    D1 / Threshold_n / MAE come from ONE fused pass per frame (consumers.evaluate, mask 0 < gt <= max_disparity); any other metric object is called
    with the reference's (estimate, gt, mask) arguments."""
    metrics = list(metrics or [])
    results: Dict[str, List[float]] = {m.name(): [] for m in metrics}
    config = pipeline.get_configuration()
    max_disp = config.max_disparity
    if hasattr(camera, "stream_image_pairs_with_gt_disparity"):
        validate_pipeline_config_wrt_camera(config, camera)
        frames_with_gt = camera.stream_image_pairs_with_gt_disparity()
    else:
        frames_with_gt = camera
    for frame_index, (left_view, right_view, gt_disparity) in enumerate(frames_with_gt):
        _check_frame_shape(config, left_view)
        gt_disparity = gt_disparity.cuda().float()
        result = pipeline.process(left_view, right_view)
        fused: Dict[float, Dict[str, float]] = {}
        mask = None
        for m in metrics:
            thr = m._threshold if isinstance(m, ThresholdMetric) else 3.0
            if type(m) in (D1Metric, ThresholdMetric, MAEMetric):
                if thr not in fused:
                    fused[thr] = consumers.evaluate(result.disparity_map, gt_disparity, max_disp, threshold=thr)
                results[m.name()].append(fused[thr][m.name()])
            else:
                if mask is None:
                    mask = (gt_disparity <= max_disp) & (gt_disparity > 0)
                results[m.name()].append(m.process(result.disparity_map, gt_disparity, mask))
        if verbose:
            print(f"Processed frame {frame_index}.")
    return reduce_metrics(results, reduction)
