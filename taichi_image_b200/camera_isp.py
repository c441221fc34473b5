"""Stateful camera ISP processor (reference: camera_isp.py).

``Camera16`` / ``Camera32`` keep the reference's constructor, ``set``, ``load_*``, ``update_metering``,
``tonemap_reinhard`` / ``tonemap_linear`` / ``tonemap_only`` and the ``metrics`` state (9 floats on the
device, moving-average semantics of camera_isp.py:376-385 including the double bounds blend).

Two ways through the same arithmetic:

* eager, stage by stage, exactly like the reference API: ``load_packed12`` returns the float RGB
  tensor, ``tonemap_*`` takes a list of them (each stage one CUDA kernel from csrc/);
* fused: ``process_packed12(frames, ...)`` runs metering + demosaic + CCM + tone map + quantisation
  straight from the packed bytes (``b200isp_process_packed12``, csrc/fused_isp.cuh) without
  materialising the CFA or the float RGB.  This is the hot path the benchmark measures.

Deviations from the reference are the ones listed in SURVEY 2.5: the configured ``bayer_pattern`` is
honoured (Q1), tone-map parameters are runtime arguments (Q13), outputs may be u8 / u16 / f16
(extension of tonemap.py:16-17).  Like the reference, ``tonemap_reinhard`` overwrites its input images
with the un-normalised map (Q6); ``process_packed12`` never touches its inputs.
"""
from __future__ import annotations

from typing import Optional, Sequence

import os

import numpy as np
import torch
from beartype import beartype

from . import _lib, bayer, interpolate, packed, types
from .dtypes import DType, as_dtype, f16, f32, u8
from .util import lerp  # noqa: F401  (re-exported like the reference module)


def moving_average(old, new, alpha):               # camera_isp.py:15-19
    if old is None:
        return new
    return (1 - alpha) * old + alpha * new


default_cc = np.array([                            # camera_isp.py:230-234
    [1.75, -0.25, -0.30],
    [-0.10, 1.40, -0.30],
    [-0.05, -0.55, 2.10],
])

_TONEMAP_CODE = {"linear": 0, "reinhard": 1, "none": 2}


def _reinhard_kernel(image, output, metering, gamma, intensity, light_adapt, color_adapt):
    """camera_isp.py:177-218 on CUDA tensors; overwrites ``image`` with the un-normalised map."""
    _lib.require_cuda(image, "reinhard_kernel")
    assert image.is_contiguous() and output.is_contiguous() and metering.dtype == torch.float32
    dt, odt = as_dtype(image.dtype), as_dtype(output.dtype)
    with torch.cuda.device(image.device):
        _lib.check(_lib.lib.b200isp_isp_reinhard(
            image.data_ptr(), dt.code, output.data_ptr(), odt.code, image.shape[0] * image.shape[1], metering.data_ptr(),
            float(gamma), float(intensity), float(light_adapt), float(color_adapt),
            _lib.workspace(image.device).data_ptr(), _lib.stream_ptr(image.device)), "isp_reinhard")


def _reinhard_batch(images, outputs, metering, gamma, intensity, light_adapt, color_adapt):
    """``_reinhard_kernel`` over a list of same-shape images: one launch per pass for the whole list"""
    dt, odt = as_dtype(images[0].dtype), as_dtype(outputs[0].dtype)
    dev = images[0].device
    with torch.cuda.device(dev):
        _lib.check(_lib.lib.b200isp_isp_reinhard_batch(
            _lib.ptr_array(images), _lib.ptr_array(outputs), len(images), dt.code, odt.code,
            images[0].shape[0] * images[0].shape[1], metering.data_ptr(), float(gamma), float(intensity),
            float(light_adapt), float(color_adapt), _lib.workspace(dev).data_ptr(), _lib.stream_ptr(dev)), "isp_reinhard_batch")


def _linear_kernel(image, output, metering, gamma):
    """camera_isp.py:220-227 -> tonemap.py:11-17 with bounds = metering[0:2]."""
    _lib.require_cuda(image, "linear_kernel")
    assert image.is_contiguous() and output.is_contiguous() and metering.dtype == torch.float32
    dt, odt = as_dtype(image.dtype), as_dtype(output.dtype)
    with torch.cuda.device(image.device):
        _lib.check(_lib.lib.b200isp_linear(image.data_ptr(), dt.code, output.data_ptr(), odt.code, image.numel(),
                                           metering.data_ptr(), float(gamma), _lib.stream_ptr(image.device)), "isp_linear")


def camera_isp(name: str, dtype=f32):
    """camera_isp.py:75 -- class factory; ``dtype`` is the ISP intermediate type (f16 or f32)."""
    isp_dtype: DType = as_dtype(dtype)
    assert isp_dtype in (f16, f32), "ISP dtype must be f16 or f32"
    torch_dtype = isp_dtype.torch

    class ISP:
        @beartype
        def __init__(self, bayer_pattern: bayer.BayerPattern,
                     scale: Optional[float] = None,
                     resize_width: int = 0,
                     moving_alpha=0.1,
                     correct_colors: bool = False,
                     white_balance: np.ndarray = np.array([1.8, 1.0, 2.1]),
                     color_correction: np.ndarray = default_cc,
                     transform: interpolate.ImageTransform = interpolate.ImageTransform.none,
                     device: torch.device = torch.device('cuda', 0),
                     metering_stride: int = 8,
                     demosaic: str = "malvar",
                     resize_size: Optional[tuple] = None,
                     reinhard_exact: Optional[bool] = None):
            """camera_isp.py:237-268.  ``demosaic="bilinear"`` (EXTENSION, north_star): 3x3 bilinear interpolation
            instead of Malvar-He-Cutler in every load / fused path of this object (``bayer_to_rgb(method=...)``)."""
            assert scale is None or resize_width == 0, "Cannot specify both scale and resize_width"
            assert resize_size is None or (scale is None and resize_width == 0), "resize_size excludes scale / resize_width"
            assert demosaic in ("malvar", "bilinear")
            # EXTENSION (BASELINE configs[4] "resize to 1920x1080"): explicit (width, height) target with per-axis scales
            # (SURVEY Q9); the reference only knows the aspect-preserving ``scale`` / ``resize_width``
            self.resize_size = None if resize_size is None else (int(resize_size[0]), int(resize_size[1]))
            self.demosaic = demosaic
            # EXTENSION: Camera32 Reinhard -> u8 runs one sweep + a u16 fixed-point map by default (u8 within 1 LSB of the exact
            # form, csrc/fused_isp.cuh); True keeps the exact max sweep + write sweep (env default: B200ISP_REINHARD_EXACT=1)
            self.reinhard_exact = (os.environ.get("B200ISP_REINHARD_EXACT", "0") == "1") if reinhard_exact is None else bool(reinhard_exact)
            self.bayer_pattern = bayer_pattern
            self.moving_alpha = moving_alpha
            self.scale = scale
            self.resize_width = resize_width
            self.transform = transform
            self.metering_stride = metering_stride
            self.correct_colors = correct_colors
            self.white_balance = white_balance
            self.color_correction = color_correction
            self.metrics = None
            self.device = device
            self.dtype = isp_dtype
            # look-ahead metering state (process_packed12(lookahead=...)): second metrics buffer, side stream,
            # the pending update for the announced next batch, completion event of the previous sweep
            self._ids_layout = False          # packed layout of the frames of the current process_packed12 call (metering included)
            self._metrics_alt = None
            self._side_stream = None
            self._lookahead = None
            self._ev_prev_sweep = None

        @beartype
        def set(self, moving_alpha: Optional[float] = None, resize_width: Optional[int] = None,
                scale: Optional[float] = None, correct_colors: Optional[bool] = None,
                white_balance: Optional[np.ndarray] = None, color_correction: Optional[np.ndarray] = None,
                transform: Optional[interpolate.ImageTransform] = None):
            """camera_isp.py:270-300"""
            if moving_alpha is not None:
                self.moving_alpha = moving_alpha
            if resize_width is not None:
                self.resize_width = resize_width
                self.scale = None
                self.resize_size = None
            if scale is not None:
                self.scale = scale
                self.resize_width = 0
                self.resize_size = None
            if transform is not None:
                self.transform = transform
            if correct_colors is not None:
                self.correct_colors = correct_colors
            if white_balance is not None:
                self.white_balance = white_balance
            if color_correction is not None:
                self.color_correction = color_correction

        # ------------------------------------------------------------ configuration helpers
        @property
        def color_correct_matrix(self) -> Optional[np.ndarray]:
            """camera_isp.py:360-369: color_correction @ diag(white_balance), or None"""
            if self.correct_colors:
                cc = np.array(self.color_correction, dtype=np.float64).copy()
                cc[:, :3] *= np.asarray(self.white_balance, dtype=np.float64)
                return cc
            return None

        def _resize_plan(self, h, w):
            """((width, height), (scale_row, scale_col)) of camera_isp.py:302-315 for an (h, w) image, or None"""
            if self.resize_width > 0:
                scale = self.resize_width / w
                return (self.resize_width, round(h * scale)), (scale, scale)
            if self.scale is not None:
                return (round(w * self.scale), round(h * self.scale)), (self.scale, self.scale)
            if self.resize_size is not None:
                wo, ho = self.resize_size
                return (wo, ho), (ho / h, wo / w)
            return None

        def resize_image(self, image):
            """camera_isp.py:302-315"""
            plan = self._resize_plan(image.shape[0], image.shape[1])
            if plan is None:
                return image
            return interpolate.resize_bilinear(image, plan[0], plan[1])

        @property
        def _resizes(self) -> bool:
            return self.resize_width > 0 or self.scale is not None or self.resize_size is not None

        # ------------------------------------------------------------ loaders (eager API)
        def _convert(self, image, mode):
            image = image.to(self.device).contiguous()
            cfa = torch.empty(image.shape, dtype=torch_dtype, device=self.device)
            with torch.cuda.device(self.device):
                _lib.check(_lib.lib.b200isp_load_convert(image.data_ptr(), cfa.data_ptr(), isp_dtype.code, image.numel(),
                                                         mode, _lib.stream_ptr(self.device)), "load_convert")
            return self._process_image(cfa)

        def load_16u(self, image):
            """camera_isp.py:82-87, :318-321: u16 -> x / 65535"""
            assert image.dtype == torch.uint16 and image.ndim == 2
            return self._convert(image, 0)

        def load_32f(self, image):
            """camera_isp.py:89-93, :328-331"""
            assert image.dtype == torch.float32 and image.ndim == 2
            return self._convert(image, 1)

        def load_16f(self, image):
            """camera_isp.py:95-99, :323-326 (annotated u16 in the reference; plain cast, no scaling)"""
            assert image.dtype == torch.uint16 and image.ndim == 2
            return self._convert(image, 2)

        def _fused_ok(self, image_data, ids_format) -> bool:
            """frames the fused sweep takes: even height >= 4, width % 8 == 0, contiguous, 4-byte aligned.  The IDS layout is
            decoded inside the sweep's row loader (csrc/fused_isp.cuh ids_sample) except by the resizing sweep."""
            h, w3 = image_data.shape
            w = w3 * 2 // 3
            return (not (ids_format and (self._resizes or self.demosaic != "malvar")) and h >= 4 and h % 2 == 0 and w >= 8 and w % 8 == 0
                    and image_data.is_contiguous() and image_data.data_ptr() % 4 == 0)

        def _ids_to_standard(self, frames):
            """IDS-layout frames that the fused sweep could otherwise take -> standard layout in a persistent scratch
            (one extra 1.5 + 1.5 B/px pass instead of the staged decode / demosaic / tone-map kernels)"""
            scratch = getattr(self, "_ids_scratch", None)
            if (scratch is None or len(scratch) < len(frames) or scratch[0].shape != frames[0].shape
                    or scratch[0].device != frames[0].device):
                scratch = self._ids_scratch = [torch.empty_like(frames[0]) for _ in frames]
            return [packed.repack12_ids(f, out=s) for f, s in zip(frames, scratch)]

        def load_packed12(self, image_data, ids_format=False):
            """camera_isp.py:333-340: decode12(scaled) + demosaic (+CCM) (+resize) -> float RGB of the ISP dtype"""
            assert image_data.dtype == torch.uint8 and image_data.ndim == 2
            image_data = image_data.to(self.device)
            if ids_format and not self._fused_ok(image_data, True) and self._fused_ok(image_data, False):
                image_data, ids_format = self._ids_to_standard([image_data])[0], False     # resizing / bilinear sweep: standard layout only
            if self._fused_ok(image_data, ids_format):
                return self._run_fused([image_data], "none", isp_dtype, None, {}, ids_format=ids_format)[0]   # resize included
            w, h = (image_data.shape[1] * 2 // 3, image_data.shape[0])
            cfa = torch.empty(h, w, dtype=torch_dtype, device=self.device)
            packed.decode12_kernel(isp_dtype, scaled=True, ids_format=ids_format)(image_data.contiguous().view(-1), cfa.view(-1))
            return self._process_image(cfa)

        def load_packed16(self, image_data):
            """camera_isp.py:342-347"""
            assert image_data.dtype == torch.uint8 and image_data.ndim == 2
            image_data = image_data.to(self.device)
            w, h = (image_data.shape[1] // 2, image_data.shape[0])
            cfa = torch.empty(h, w, dtype=torch_dtype, device=self.device)
            packed.decode16_kernel(isp_dtype, scaled=True)(image_data.contiguous().view(-1), cfa.view(-1))
            return self._process_image(cfa)

        def load_packed10(self, image_data):
            """EXTENSION (SURVEY 8f-4): MIPI RAW10 frames, (H, 5 W / 4) bytes -- decoded to the ISP dtype scaled by 1 / 1023
            (``packed.decode10``), then the path of ``load_packed16``"""
            assert image_data.dtype == torch.uint8 and image_data.ndim == 2 and image_data.shape[1] % 5 == 0
            image_data = image_data.to(self.device)
            w, h = (image_data.shape[1] * 4 // 5, image_data.shape[0])
            cfa = torch.empty(h, w, dtype=torch_dtype, device=self.device)
            packed.decode10_kernel(isp_dtype, scaled=True)(image_data.contiguous().view(-1), cfa.view(-1))
            return self._process_image(cfa)

        def _process_image(self, cfa):
            """camera_isp.py:371-373 (with the configured pattern, SURVEY Q1)"""
            rgb = bayer.bayer_to_rgb(cfa, self.bayer_pattern, correct_colors=self.color_correct_matrix, method=self.demosaic)
            return self.resize_image(rgb)

        # ------------------------------------------------------------ metering
        def _metrics_and_alpha(self):
            """camera_isp.py:376-385: first call blends from zeros with t = 0, later t = 1 - moving_alpha"""
            if self.metrics is None:
                self.metrics = torch.zeros(9, dtype=torch.float32, device=self.device)
                return 0.0
            return 1.0 - float(self.moving_alpha)

        def update_metering(self, images: Sequence[torch.Tensor]):
            """camera_isp.py:376-385 over stack([im[::stride, ::stride] for im in images])"""
            assert len(images) >= 1
            assert len(images) <= _lib.MAX_FRAMES, f"at most {_lib.MAX_FRAMES} images per metering call"
            shape = images[0].shape
            for im in images:
                _lib.require_cuda(im, "update_metering")
                assert im.shape == shape and im.dtype == torch_dtype and im.is_contiguous(), \
                    "metering needs same-shape contiguous images of the ISP dtype"
            alpha = self._metrics_and_alpha()
            with torch.cuda.device(self.device):
                _lib.check(_lib.lib.b200isp_metering_update(
                    _lib.ptr_array(images), len(images), isp_dtype.code, shape[0], shape[1], int(self.metering_stride),
                    alpha, self.metrics.data_ptr(), _lib.workspace(self.device).data_ptr(),
                    _lib.stream_ptr(self.device)), "metering_update")

        # ------------------------------------------------------------ metering split for multi-GPU shared exposure
        # (distributed.SharedExposure; include/b200isp.h "multi-GPU shared exposure").  ``source`` is either a list
        # of packed12 frames (uint8, 2-D: the fused sampler) or a list of ISP-dtype RGB images.
        def _meter_source(self, source):
            source = list(source)
            packed12 = source[0].dtype == torch.uint8 and source[0].ndim == 2
            shape = source[0].shape
            for t in source:
                _lib.require_cuda(t, "metering")
                assert t.shape == shape and t.is_contiguous(), "metering needs same-shape contiguous tensors"
                assert packed12 or t.dtype == torch_dtype, "metering images must have the ISP dtype"
            assert 1 <= len(source) <= _lib.MAX_FRAMES
            return source, packed12

        def meter_phase1(self, source) -> torch.Tensor:
            """{min, max} over this rank's metering samples -> 2 floats on the device"""
            source, packed12 = self._meter_source(source)
            rec = torch.empty(2, dtype=torch.float32, device=self.device)
            ws, st = _lib.workspace(self.device).data_ptr(), _lib.stream_ptr(self.device)
            with torch.cuda.device(self.device):
                if packed12:
                    p = self._fused_params(source, "linear", u8, {}, update_metering=True)
                    _lib.check(_lib.lib.b200isp_meter_packed12_phase1(_lib.ptr_array(source), len(source), p,
                                                                       rec.data_ptr(), ws, st), "meter_packed12_phase1")
                else:
                    h, w = source[0].shape[:2]
                    _lib.check(_lib.lib.b200isp_metering_phase1(_lib.ptr_array(source), len(source), isp_dtype.code, h, w,
                                                                 int(self.metering_stride), rec.data_ptr(), ws, st),
                               "metering_phase1")
            return rec

        def meter_phase2(self, source, gathered1: torch.Tensor, alpha: float) -> torch.Tensor:
            """statistics of this rank's samples w.r.t. the joint blended bounds -> 8 floats on the device"""
            source, packed12 = self._meter_source(source)
            assert gathered1.dtype == torch.float32 and gathered1.is_contiguous() and gathered1.numel() % 2 == 0
            world = gathered1.numel() // 2
            rec = torch.empty(8, dtype=torch.float32, device=self.device)
            ws, st = _lib.workspace(self.device).data_ptr(), _lib.stream_ptr(self.device)
            with torch.cuda.device(self.device):
                if packed12:
                    p = self._fused_params(source, "linear", u8, {}, update_metering=True, alpha=alpha)
                    _lib.check(_lib.lib.b200isp_meter_packed12_phase2(
                        _lib.ptr_array(source), len(source), p, gathered1.data_ptr(), world, self.metrics.data_ptr(),
                        rec.data_ptr(), ws, st), "meter_packed12_phase2")
                else:
                    h, w = source[0].shape[:2]
                    _lib.check(_lib.lib.b200isp_metering_phase2(
                        _lib.ptr_array(source), len(source), isp_dtype.code, h, w, int(self.metering_stride),
                        gathered1.data_ptr(), world, float(alpha), self.metrics.data_ptr(), rec.data_ptr(), ws, st),
                        "metering_phase2")
            return rec

        def meter_finalize(self, gathered1: torch.Tensor, gathered2: torch.Tensor, alpha: float, out: Optional[torch.Tensor] = None):
            """out (default: metrics, in place) = lerp(alpha, joint statistics of all ranks, metrics)   (camera_isp.py:164-166)"""
            world = gathered1.numel() // 2
            assert gathered2.numel() == 8 * world and gathered2.is_contiguous() and gathered1.is_contiguous()
            out = self.metrics if out is None else out
            with torch.cuda.device(self.device):
                _lib.check(_lib.lib.b200isp_metering_finalize(gathered1.data_ptr(), gathered2.data_ptr(), world, float(alpha),
                                                               self.metrics.data_ptr(), out.data_ptr(),
                                                               _lib.stream_ptr(self.device)), "metering_finalize")

        def meter_packed12(self, frames, alpha: float, out: Optional[torch.Tensor] = None, cooperative: bool = True):
            """camera_isp.py:376-385 straight from packed12 frames on the current stream:
            out (default: metrics, in place) = lerp(alpha, statistics(frames), metrics)"""
            out = self.metrics if out is None else out
            p = self._fused_params(frames, "linear", u8, {}, update_metering=True, alpha=alpha)
            with torch.cuda.device(self.device):
                _lib.check(_lib.lib.b200isp_meter_packed12(
                    _lib.ptr_array(frames), len(frames), p, self.metrics.data_ptr(), out.data_ptr(), int(cooperative),
                    _lib.workspace(self.device).data_ptr(), _lib.stream_ptr(self.device)), "meter_packed12")

        def meter_packed12_shared(self, frames, alpha: float, peer, out: Optional[torch.Tensor] = None):
            """``meter_packed12`` jointly with the other ranks of ``peer`` (distributed.PeerExchange): two launches, the
            record exchanges over NVLink run inside the metering kernels; all ranks end with bit-identical metrics"""
            out = self.metrics if out is None else out
            p = self._fused_params(frames, "linear", u8, {}, update_metering=True, alpha=alpha)
            with torch.cuda.device(self.device):
                _lib.check(_lib.lib.b200isp_meter_packed12_shared(
                    _lib.ptr_array(frames), len(frames), p, peer._peers, peer.world, peer.rank, self.metrics.data_ptr(),
                    out.data_ptr(), _lib.workspace(self.device).data_ptr(), _lib.stream_ptr(self.device)), "meter_packed12_shared")

        # ------------------------------------------------------------ percentile histogram (EXTENSION, north_star)
        def metering_histogram(self, bins: int = 256) -> torch.Tensor:
            """Luminance histogram (``bins`` int32 counts over [0, 1]) of the samples of the LAST fused metering
            (``process_packed12`` / ``meter_packed12``): the same ``[::stride, ::stride]`` RGB samples of all frames the
            reference's statistics are computed from (camera_isp.py:168-170).  No reference counterpart."""
            cache, n = getattr(self, "_meter_cache", None), getattr(self, "_meter_n", 0)
            assert cache is not None and n > 0, "no fused metering has run yet"
            hist = torch.empty(bins, dtype=torch.int32, device=self.device)
            with torch.cuda.device(self.device):
                _lib.check(_lib.lib.b200isp_sample_histogram(cache.data_ptr(), n, int(bins), hist.data_ptr(),
                                                             _lib.stream_ptr(self.device)), "sample_histogram")
            return hist

        def metering_percentiles(self, percents=(1.0, 50.0, 99.0), bins: int = 256) -> torch.Tensor:
            """luminance percentiles (upper bin edges in [0, 1]) from ``metering_histogram``; stays on the device"""
            hist = self.metering_histogram(bins)
            pct = torch.tensor([float(p) for p in percents], dtype=torch.float32, device=self.device)
            out = torch.empty(len(pct), dtype=torch.float32, device=self.device)
            with torch.cuda.device(self.device):
                _lib.check(_lib.lib.b200isp_histogram_percentiles(hist.data_ptr(), int(bins), pct.data_ptr(), len(pct), out.data_ptr(),
                                                                  _lib.stream_ptr(self.device)), "histogram_percentiles")
            return out

        # ------------------------------------------------------------ tone mapping (eager API)
        def tonemap_only(self, image, metrics, gamma, intensity, light_adapt, color_adapt):
            """camera_isp.py:387-390"""
            output = torch.empty(image.shape, dtype=torch.uint8, device=self.device)
            _reinhard_kernel(image, output, metrics, gamma, intensity, light_adapt, color_adapt)
            return interpolate.transform(output, self.transform)

        @beartype
        def tonemap_reinhard(self, images: list[torch.Tensor], gamma: float = 1.0, intensity: float = 1.0,
                             light_adapt: float = 1.0, color_adapt: float = 0.0, dtype=u8, update_metering: bool = True):
            """camera_isp.py:394-403 (``dtype``: u8 like the reference, or u16 / f16; ``update_metering=False``:
            the caller -- distributed.SharedExposure -- has already updated ``self.metrics``)"""
            out_dtype = as_dtype(dtype)
            if update_metering:
                self.update_metering(images)
            outputs = [torch.empty(image.shape, dtype=out_dtype.torch, device=self.device) for image in images]
            same = all(im.shape == images[0].shape and im.dtype == images[0].dtype and im.is_cuda and im.is_contiguous()
                       for im in images)
            if same and 1 < len(images) <= _lib.MAX_FRAMES:
                _reinhard_batch(images, outputs, self.metrics, gamma, intensity, light_adapt, color_adapt)
            else:
                for output, image in zip(outputs, images):
                    _reinhard_kernel(image, output, self.metrics, gamma, intensity, light_adapt, color_adapt)
            return [interpolate.transform(output, self.transform) for output in outputs]

        @beartype
        def tonemap_linear(self, images: list[torch.Tensor], gamma: float = 1.0, dtype=u8, update_metering: bool = True):
            """camera_isp.py:405-413"""
            out_dtype = as_dtype(dtype)
            if update_metering:
                self.update_metering(images)
            outputs = [torch.empty(image.shape, dtype=out_dtype.torch, device=self.device) for image in images]
            for output, image in zip(outputs, images):
                _linear_kernel(image, output, self.metrics, gamma)
            return [interpolate.transform(output, self.transform) for output in outputs]

        # ------------------------------------------------------------ fused path
        def _param_block(self, h, w, tonemap, out_dtype, tm, yuv420=False, ids_format=None, flip=0, out_pitch=0):
            """b200isp_fused_params (include/b200isp.h) describing the images and the tone map of a call on (h, w) frames;
            no buffer attached"""
            p = _lib.FusedParams()
            p.height, p.width, p.pattern = h, w, self.bayer_pattern.value
            p.isp_dtype, p.out_dtype, p.tonemap = isp_dtype.code, out_dtype.code, _TONEMAP_CODE[tonemap]
            ccm = self.color_correct_matrix
            p.has_ccm = 0 if ccm is None else 1
            for i, v in enumerate((np.zeros(9) if ccm is None else ccm.reshape(-1))):
                p.ccm[i] = float(v)
            p.gamma = float(tm.get("gamma", 1.0))
            p.intensity = float(tm.get("intensity", 1.0))
            p.light_adapt = float(tm.get("light_adapt", 1.0))
            p.color_adapt = float(tm.get("color_adapt", 0.0))
            p.metering_stride = int(self.metering_stride)
            p.demosaic = 1 if self.demosaic == "bilinear" else 0
            p.out_yuv420 = int(bool(yuv420))
            p.ids_layout = int(bool(self._ids_layout if ids_format is None else ids_format))
            p.flip, p.out_pitch = int(flip), int(out_pitch)
            if tonemap == "reinhard" and self.reinhard_exact:
                p.reinhard_mode = 1
            plan = self._resize_plan(h, w)
            if plan is not None:                 # resize fused into the pass (demosaic + bilinear gather)
                (wo, ho), (sr, sc) = plan
                p.out_height, p.out_width, p.scale_r, p.scale_c = int(ho), int(wo), float(sr), float(sc)
                p.resize_gather = int(os.environ.get("B200ISP_RESIZE_GATHER", "0"))        # testing / profiling knob
            return p

        def _fused_params(self, frames, tonemap, out_dtype, tm, update_metering=False, alpha=0.0, rows_per_task=0,
                          profile_events=None, yuv420=False, ids_format=None, flip=0, out_pitch=0):
            """b200isp_fused_params for a list of same-shape packed12 frames (include/b200isp.h), with the buffers the call uses"""
            h, w3 = frames[0].shape
            p = self._param_block(h, w3 * 2 // 3, tonemap, out_dtype, tm, yuv420, ids_format, flip, out_pitch)
            p.alpha = float(alpha)
            p.update_metering, p.rows_per_task = int(update_metering), int(rows_per_task)
            if update_metering:                  # scratch for the phase-1 samples (re-read by phase 2)
                ho, wo = (p.out_height, p.out_width) if p.out_height > 0 else (p.height, p.width)
                stride = max(int(self.metering_stride), 1)
                need = len(frames) * (-(-ho // stride)) * (-(-wo // stride)) * 12
                cache = getattr(self, "_meter_cache", None)
                if cache is None or cache.numel() < need or cache.device != torch.device(self.device):
                    if cache is not None:
                        torch.cuda.synchronize(self.device)      # a look-ahead metering on the side stream may still use it
                    cache = self._meter_cache = torch.empty(need, dtype=torch.uint8, device=self.device)
                p.meter_cache, p.meter_cache_bytes = cache.data_ptr(), cache.numel()
                self._meter_n = need // 12
            # scratch of the one-sweep Reinhard forms, sized by the library that chooses the form (csrc/fused_isp.cuh
            # reinhard_plan); none where the call runs the exact max sweep + write sweep
            need = _lib.lib.b200isp_reinhard_scratch_bytes(p, len(frames))
            if need:
                sc = getattr(self, "_reinhard_scratch", None)
                if sc is None or sc.numel() < need or sc.device != torch.device(self.device):
                    sc = self._reinhard_scratch = torch.empty(need, dtype=torch.uint8, device=self.device)
                p.reinhard_scratch, p.reinhard_scratch_bytes = sc.data_ptr(), sc.numel()
            if profile_events is not None:      # (start, stop) torch.cuda.Event pair, see bench.py
                p.profile_start, p.profile_stop = profile_events[0].cuda_event, profile_events[1].cuda_event
            return p

        def _fused_flip(self, height, tonemap, out_dtype, gamma, color_adapt, ids_format=False, yuv420=False):
            """b200isp_fused_params.flip code of ``self.transform`` when the fused call applies the transform itself, else 0
            (the tiled transform kernel then runs on the results)"""
            flip = 0
            if not self._resizes and not yuv420 and self.demosaic == "malvar":
                T = interpolate.ImageTransform
                flip = {T.flip_horiz: 1, T.flip_vert: 2, T.rotate_180: 3, T.transpose: 4, T.rotate_270: 5, T.rotate_90: 6,
                        T.transverse: 7}.get(self.transform, 0)
                # Transposing transforms (rotate_90 is the rig script's default): the one-sweep Reinhard -> u8 forms turn the
                # image in their element-wise normalise pass (csrc/fused_isp.cuh reinhard_out_transposed_kernel: shared-memory
                # tile, 384-byte output pieces) -- no transform kernel, no extra 3 + 3 B/px.  The library accepts bit 2 exactly
                # when it asks for a scratch for such a form; no rule of that query reads the width, so any valid width does.
                # Every other call runs the transform kernel on its results.
                if flip & 4:
                    p = self._param_block(height, 8, tonemap, out_dtype, dict(gamma=gamma, color_adapt=color_adapt),
                                          yuv420, bool(ids_format), flip)
                    if not _lib.lib.b200isp_reinhard_scratch_bytes(p, 1):
                        flip = 0
            return flip

        def _run_fused(self, frames, tonemap, out_dtype, out, tm, update_metering=False, alpha=0.0, rows_per_task=0,
                       profile_events=None, yuv420=False, ids_format=None, flip=0):
            h, w3 = frames[0].shape
            w = w3 * 2 // 3
            if yuv420 and not (isp_dtype == f16 and tonemap == "reinhard" and not self._resizes):
                # no YUV epilogue for this path: RGB8 into a persistent scratch, then the stand-alone RGB -> planar YUV 4:2:0
                # kernel (csrc/yuv420.cu) on the device -- bit-identical to color.rgb_yuv420_image of the RGB result; the
                # host only ever sees 1.5 bytes per pixel
                return self._run_fused_yuv_two_step(frames, tonemap, out_dtype, out, tm, update_metering, alpha, rows_per_task,
                                                    profile_events)
            plan = self._resize_plan(h, w)
            if plan is not None:
                w, h = plan[0]
            oshape = (h * 3 // 2, w) if yuv420 else (h, w, 3)       # planar YUV 4:2:0: color/yuv_420.py:95-118
            if flip & 4:
                oshape = (w, h, 3)                                  # transposing transform applied by the normalise pass
            out_pitch = 0
            if out is None:
                out = [torch.empty(oshape, dtype=out_dtype.torch, device=self.device) for _ in frames]
            else:
                # dense frames, or equally pitched tiles of a larger image (rig.GridOutput: the camera grid of
                # scripts/tonemap_scan.py:91-100 written in place by the sweep)
                assert len(out) == len(frames)
                pitch = out[0].stride(0) if out[0].ndim == 3 else 0
                for o in out:
                    assert tuple(o.shape) == oshape and o.dtype == out_dtype.torch and o.is_cuda
                    assert o.is_contiguous() or (o.ndim == 3 and o.stride() == (pitch, 3, 1) and pitch >= 3 * oshape[1]), \
                        "outputs must be contiguous or row-pitched (H, W, 3) views"
                if not out[0].is_contiguous():
                    assert plan is None and not yuv420, "pitched outputs need the plain RGB sweep (no resize, no YUV)"
                    out_pitch = pitch
            p = self._fused_params(frames, tonemap, out_dtype, tm, update_metering, alpha, rows_per_task, profile_events, yuv420,
                                   ids_format, flip, out_pitch=out_pitch)
            metrics_ptr = 0 if self.metrics is None else self.metrics.data_ptr()
            with torch.cuda.device(self.device):
                _lib.check(_lib.lib.b200isp_process_packed12(
                    _lib.ptr_array(frames), _lib.ptr_array(out), len(frames), p, metrics_ptr,
                    _lib.workspace(self.device).data_ptr(), _lib.stream_ptr(self.device)), "process_packed12")
            return out

        def _run_fused_yuv_two_step(self, frames, tonemap, out_dtype, out, tm, update_metering, alpha, rows_per_task, profile_events):
            from .color.yuv_420 import YCrCb_T_bgr, _mat9
            assert out_dtype == u8, "yuv420 output is u8"
            h, w = frames[0].shape[0], frames[0].shape[1] * 2 // 3
            plan = self._resize_plan(h, w)
            ho, wo = (h, w) if plan is None else (plan[0][1], plan[0][0])
            assert ho % 2 == 0 and wo % 2 == 0, "yuv420 output needs even output dimensions"
            rgb = getattr(self, "_yuv_rgb_scratch", None)
            if rgb is None or len(rgb) < len(frames) or tuple(rgb[0].shape) != (ho, wo, 3) or rgb[0].device != torch.device(self.device):
                rgb = self._yuv_rgb_scratch = [torch.empty((ho, wo, 3), dtype=torch.uint8, device=self.device) for _ in frames]
            rgb = self._run_fused(frames, tonemap, out_dtype, rgb[:len(frames)], tm, update_metering, alpha, rows_per_task, profile_events)
            if out is None:
                out = [torch.empty((ho * 3 // 2, wo), dtype=torch.uint8, device=self.device) for _ in frames]
            mat = _mat9(YCrCb_T_bgr)
            with torch.cuda.device(self.device):
                for r, o in zip(rgb, out):
                    assert tuple(o.shape) == (ho * 3 // 2, wo) and o.dtype == torch.uint8 and o.is_contiguous() and o.is_cuda
                    _lib.check(_lib.lib.b200isp_rgb_yuv420(r.data_ptr(), u8.code, o.data_ptr(), u8.code, ho, wo, mat,
                                                           _lib.stream_ptr(self.device)), "rgb_yuv420")
            return out

        def process_packed12(self, frames: Sequence[torch.Tensor], tonemap: str = "reinhard", gamma: float = 1.0,
                             intensity: float = 1.0, light_adapt: float = 1.0, color_adapt: float = 0.0,
                             dtype=u8, ids_format: bool = False, out: Optional[list] = None,
                             rows_per_task: int = 0, profile_events=None, update_metering: bool = True,
                             lookahead: Optional[Sequence[torch.Tensor]] = None, meter_fn=None, yuv420: bool = False):
            """Fused equivalent of ``[load_packed12(f) for f in frames]`` followed by
            ``tonemap_reinhard`` / ``tonemap_linear`` (camera_isp.py:333-340, :376-413): joint metering of
            all frames with the moving-average update of ``self.metrics``, then one sweep per frame.
            Returns the list of tone-mapped (H, W, 3) images (transformed if ``self.transform`` is set).
            A resizing ISP runs the fused demosaic + bilinear-resize gather (csrc/fused_resize.cu: the metering and the tone
            map then see the resized image, like the reference).  Falls back to the staged CUDA kernels when the frames
            have a width that is not a multiple of 8 -- never to the CPU.

            ``lookahead``: the frames of the NEXT call (a camera stream knows them: they are being captured / copied
            while this batch is processed).  Their metering update -- which only depends on this call's metrics --
            is then issued on a side stream and runs under this batch's sweep; the next call finds it done.  The
            announced tensors must not be modified before that call.  Results are identical to calling without it.
            ``meter_fn(frames, alpha, out, cooperative)``: replaces the local metering (distributed.SharedExposure).

            ``yuv420=True`` (u8, fused frames only): every output is the planar YUV 4:2:0 image
            ``color.rgb_yuv420_image`` would make of the RGB8 result -- ``(3H/2, W)`` u8, bit-identical.  Camera16 +
            Reinhard writes it directly from the normalise pass (no RGB image at all); every other path runs the RGB8
            sweep into a device scratch followed by the stand-alone conversion kernel -- the host sees 1.5 B/px either way."""
            assert tonemap in ("linear", "reinhard")
            out_dtype = as_dtype(dtype)
            if yuv420:
                assert out_dtype == u8, "yuv420 output is u8"
                assert self.transform == interpolate.ImageTransform.none, "yuv420 output cannot be transformed"
            frames = [f.to(self.device) for f in frames]
            assert 1 <= len(frames) <= _lib.MAX_FRAMES, f"1..{_lib.MAX_FRAMES} frames per call"
            shape = frames[0].shape
            assert all(f.shape == shape and f.dtype == torch.uint8 and f.ndim == 2 for f in frames)
            if ids_format and not all(self._fused_ok(f, True) for f in frames) and all(self._fused_ok(f, False) for f in frames):
                # IDS layout + resizing / bilinear sweep: re-pack into the standard layout (scratch reused by every call, hence no look-ahead)
                frames, ids_format, lookahead = self._ids_to_standard(frames), False, None
                self._lookahead = None
            fused = all(self._fused_ok(f, ids_format) for f in frames)
            self._ids_layout = bool(ids_format) and fused      # every _fused_params of this call (sweep, metering) decodes IDS
            assert fused or not yuv420, "yuv420 output needs frames the fused sweep accepts (width % 8 == 0)"
            if not fused:
                images = [self.load_packed12(f, ids_format) for f in frames]
                if meter_fn is not None and update_metering:      # distributed.SharedExposure: joint metering of all ranks
                    meter_fn(images, None, None, True)
                    update_metering = False
                if tonemap == "linear":
                    res = self.tonemap_linear(images, gamma=float(gamma), dtype=out_dtype, update_metering=update_metering)
                else:
                    res = self.tonemap_reinhard(images, gamma=float(gamma), intensity=float(intensity),
                                                light_adapt=float(light_adapt), color_adapt=float(color_adapt),
                                                dtype=out_dtype, update_metering=update_metering)
                if out is not None:                # staged kernels allocate their own results: honour the caller's buffers
                    assert len(out) == len(res) and all(o.shape == r.shape and o.dtype == r.dtype for o, r in zip(out, res)), \
                        "out= buffers must have the shape / dtype of the (resized, transformed) results"
                    for o, r in zip(out, res):
                        o.copy_(r)
                    return list(out)
                return res
            tm = dict(gamma=gamma, intensity=intensity, light_adapt=light_adapt, color_adapt=color_adapt)
            # the transforms of interpolate.py:36-56 inside the call (no extra pass): the flips by the sweep's store
            # (csrc/fused_isp.cuh store_out), the transposing ones by the normalise pass of the one-sweep Reinhard -> u8 forms;
            # otherwise (flip == 0) the tiled transform kernel runs on the results
            flip = self._fused_flip(shape[0], tonemap, out_dtype, gamma, color_adapt, ids_format, yuv420)
            if yuv420 or flip or self.transform == interpolate.ImageTransform.none:
                finish = lambda outs: outs
            elif out is None:
                finish = lambda outs: [interpolate.transform(o, self.transform) for o in outs]
            else:                          # transform kernel after the sweep, results into the caller's (transformed-shape) buffers
                user_out, out = list(out), None
                def finish(outs):
                    res = [interpolate.transform(o, self.transform) for o in outs]
                    assert len(res) == len(user_out) and all(u.shape == r.shape and u.dtype == r.dtype for u, r in zip(user_out, res)), \
                        "out= buffers must have the shape / dtype of the transformed results"
                    for u, r in zip(user_out, res):
                        u.copy_(r)
                    return user_out
            pipelined = update_metering and (lookahead is not None or self._lookahead is not None or meter_fn is not None)
            if not pipelined:
                alpha = self._metrics_and_alpha() if update_metering else 0.0
                assert self.metrics is not None, "update_metering=False needs metrics from an earlier call"
                outputs = self._run_fused(frames, tonemap, out_dtype, out, tm, update_metering=update_metering, alpha=alpha,
                                          rows_per_task=rows_per_task, profile_events=profile_events, yuv420=yuv420, flip=flip)
                return finish(outputs)

            # ---- look-ahead pipeline: metering(k+1) on the side stream under sweep(k)
            meter = meter_fn if meter_fn is not None else self.meter_packed12
            main = torch.cuda.current_stream(self.device)
            with torch.cuda.device(self.device):
                # Everything the side stream touches exists BEFORE any work of this call is enqueued: a buffer
                # created later would be initialised on the main stream behind the sweep, i.e. after the side-stream
                # metering that writes it.  (torch.empty: the metering kernels write all nine floats.)
                if self._side_stream is None:
                    # high priority: the metering CTAs take SM slots ahead of the sweep's not-yet-dispatched
                    # CTAs (an earlier-launched grid otherwise keeps every freed slot until its tail)
                    self._side_stream = torch.cuda.Stream(self.device, priority=-1)
                if self._metrics_alt is None:
                    self._metrics_alt = torch.empty(9, dtype=torch.float32, device=self.device)
            key = lambda fs: tuple((f.data_ptr(), tuple(f.shape)) for f in fs)
            pending, self._lookahead = self._lookahead, None
            if pending is not None and pending["key"] == key(frames):
                main.wait_event(pending["event"])                      # metrics for this batch were computed ahead
                self.metrics, self._metrics_alt = pending["out"], self.metrics
                ready = pending["event"]
            else:
                if pending is not None:
                    # wrong announcement: the stale side-stream metering shares the sample cache, the workspace and
                    # (shared exposure) the mailbox sequence with the metering issued now -> let it drain first
                    main.wait_event(pending["event"])
                alpha = self._metrics_and_alpha()
                meter(frames, alpha, None, True)                       # in place, on the main stream
                ready = torch.cuda.Event()
                ready.record(main)
            outputs = self._run_fused(frames, tonemap, out_dtype, out, tm, update_metering=False,
                                      rows_per_task=rows_per_task, profile_events=profile_events, yuv420=yuv420, flip=flip)
            ev_sweep = torch.cuda.Event()
            ev_sweep.record(main)
            if lookahead is not None:
                nxt = [f.to(self.device) for f in lookahead]
                if all(self._fused_ok(f, ids_format) for f in nxt):
                    with torch.cuda.device(self.device):
                        side = self._side_stream
                        side.wait_event(ready)                         # needs this batch's metrics ...
                        if self._ev_prev_sweep is not None:
                            side.wait_event(self._ev_prev_sweep)       # ... and overwrites the buffer the previous sweep read
                        with torch.cuda.stream(side):
                            meter(nxt, 1.0 - float(self.moving_alpha), self._metrics_alt, False)
                            done = torch.cuda.Event()
                            done.record(side)
                    self._lookahead = dict(key=key(nxt), event=done, out=self._metrics_alt, frames=nxt)
            self._ev_prev_sweep = ev_sweep
            return finish(outputs)

    ISP.reinhard_kernel = staticmethod(_reinhard_kernel)     # camera_isp.py:415-416
    ISP.linear_kernel = staticmethod(_linear_kernel)
    ISP.__qualname__ = name
    ISP.__name__ = name
    return ISP


Camera16 = camera_isp("Camera16", f16)     # camera_isp.py:422-423
Camera32 = camera_isp("Camera32", f32)
