"""Tracker-side drop-in for ``lib/test/tracker/vit_dist.py``: ``get_tracker_class()`` returns a class
with the reference's plugin surface - ``__init__(params, dataset_name)``, ``initialize(image, info)``,
``track(image, info)`` -> ``{'target_bbox': [x, y, w, h], 'confidence': ...}`` - whose per-frame work
(crop, resize, normalise, stem, ViT blocks, head, Hann window, arg-max, box decode) runs in
libvittrack_b200's sm_100a kernels.  Only the two scalar box transforms the reference performs on
Python floats after ``.tolist()`` (``map_box_back``, ``clip_box``) stay on the host, so that the
returned list holds exactly the Python numbers the reference would return."""
from __future__ import annotations

import math
import os
from typing import Optional

import numpy as np
import torch

from .engine import yuv420_frame_hw, yuv_format
from .model import build_ostrack_dist
from .sequences import crop_rect
from .weights import load_checkpoint


def even_rect(rect, H: int, W: int) -> tuple:
    """``rect`` = (ya, yb, xa, xb) widened to even bounds inside an even H x W frame: the rectangle vt_upload_yuv420_rect converts
    (a 2x2 luma block shares one chroma sample)."""
    ya, yb, xa, xb = rect
    return ya & ~1, min(H, (yb + 1) & ~1), xa & ~1, min(W, (xb + 1) & ~1)


def clip_box(box: list, H, W, margin=0):
    """lib/utils/box_ops.py:97-106, same arithmetic on Python scalars."""
    x1, y1, w, h = box
    x2, y2 = x1 + w, y1 + h
    x1 = min(max(0, x1), W - margin)
    x2 = min(max(margin, x2), W)
    y1 = min(max(0, y1), H - margin)
    y2 = min(max(margin, y2), H)
    w = max(margin, x2 - x1)
    h = max(margin, y2 - y1)
    return [x1, y1, w, h]


class BaseTracker:
    """Plugin base class (lib/test/tracker/basetracker.py:10-36) without the visdom debug UI."""

    def __init__(self, params):
        self.params = params
        self.visdom = None

    def predicts_segmentation_mask(self):
        return False

    def initialize(self, image, info: dict) -> dict:
        raise NotImplementedError

    def track(self, image, info: dict = None) -> dict:
        raise NotImplementedError


class Vit_dist(BaseTracker):
    def __init__(self, params, dataset_name=None):
        super().__init__(params)
        self.cfg = params.cfg
        depth = int(getattr(params, "depth", getattr(params.cfg.MODEL.BACKBONE, "DEPTH", 3)))
        network = build_ostrack_dist(params.cfg, depth=depth, blocks_impl=getattr(params, "blocks_impl", "tcgen05"))
        ckpt = getattr(params, "checkpoint", None)
        state_dict = getattr(params, "state_dict", None)         # in-memory alternative to a checkpoint file
        if state_dict is None:
            if not ckpt or not os.path.isfile(ckpt):
                raise FileNotFoundError(f"checkpoint not found: {ckpt} (set params.checkpoint or params.state_dict)")
            state_dict = load_checkpoint(ckpt)
        network.load_state_dict(state_dict, strict=False)
        self.network = network.cuda()
        self.network.eval()
        self.engine = self.network.engine
        self.state = None
        self.feat_sz = self.cfg.TEST.SEARCH_SIZE // self.cfg.MODEL.BACKBONE.STRIDE
        self.debug = getattr(params, "debug", 0)
        self.frame_id = 0
        self.save_all_boxes = getattr(params, "save_all_boxes", False)
        if self.save_all_boxes:
            raise NotImplementedError("save_all_boxes is not supported (it also fails in the reference: "
                                      "cfg.MODEL.NUM_OBJECT_QUERIES is undefined for vit_dist)")
        dev = self.engine.device
        self._dev = dev
        self._frame_dev: Optional[torch.Tensor] = None
        self._frame_pin: Optional[torch.Tensor] = None
        self._hw = (-1, -1)
        self._hw_dev = torch.zeros((1, 2), dtype=torch.int32, device=dev)
        self._off_dev = torch.zeros((1,), dtype=torch.int64, device=dev)
        self._box_pin = self._pinned(torch.zeros((1, 4), dtype=torch.float64))
        self._box_np = self._box_pin.numpy()                      # the same memory, written without tensor indexing
        self._box_dev = torch.zeros((1, 4), dtype=torch.float64, device=dev)
        self._out_dev = torch.zeros((13,), dtype=torch.float64, device=dev)
        self._out_pin = self._pinned(torch.zeros((13,), dtype=torch.float64))
        self._out_boxes = self._out_dev[:5].view(1, 5)
        self._out_detail = self._out_dev[5:].view(1, 8)
        self._graph, self._graph_key = None, None
        # params.frame_format: "rgb" (H x W x 3, the reference's input) or a YUV 4:2:0 layout as decoders hand it out, "nv12" or
        # "i420" ((H*3/2) x W, as cv2.cvtColor takes it), converted on the device bit for bit as cv2.cvtColor(COLOR_YUV2RGB_*) would
        self.frame_format = getattr(params, "frame_format", "rgb")
        if self.frame_format != "rgb":
            yuv_format(self.frame_format)

    # ------------------------------------------------------------------------------------------
    def _pinned(self, t: torch.Tensor) -> torch.Tensor:
        return t.pin_memory() if self._dev.type == "cuda" else t

    def _sync(self) -> None:
        if self._dev.type == "cuda":
            torch.cuda.current_stream(self._dev).synchronize()

    def _upload(self, image: np.ndarray, box, factor: float):
        """Stage the rows of ``image`` the crop will read into the device frame buffer (as RGB, whatever the frame format)."""
        yuv = self.frame_format != "rgb"
        if yuv:
            if not isinstance(image, np.ndarray):
                raise ValueError(f"image must be a ({self.frame_format}) numpy array")
            H, W = yuv420_frame_hw(image)
        else:
            if image.dtype != np.uint8 or image.ndim != 3 or image.shape[2] != 3:
                raise ValueError("image must be HxWx3 uint8")
            H, W, _ = image.shape
        image = np.ascontiguousarray(image)
        if (H, W) != self._hw:
            # zero-filled: the crop kernels read the first pixels of a row with weight 0 for taps in the padding
            self._frame_dev = torch.zeros((H * W * 3,), dtype=torch.uint8, device=self._dev)
            self._frame_pin = self._pinned(torch.empty((H * W * 3,), dtype=torch.uint8))
            self._frame_stage = torch.empty((H * W * 3,), dtype=torch.uint8, device=self._dev)
            self._hw_dev.copy_(torch.tensor([[H, W]], dtype=torch.int32))
            self._hw = (H, W)
        x, y, w, h = [float(v) for v in box]
        crop_sz = math.ceil(math.sqrt(w * h) * factor)          # processing_utils.py:30
        if crop_sz < 1:
            raise Exception('Too small bounding box.')          # processing_utils.py:32-33
        # only the rectangle sample_target slices (processing_utils.py:34-48: im[y1:y2, x1:x2]) is staged and sent (crop_rect)
        rect = crop_rect(box, factor, H, W)
        if rect is None:
            raise ValueError("crop lies outside the image (undefined in the reference)")
        ya, yb, xa, xb = rect
        if yuv:
            # the even-widened rectangle (a superset of crop_rect) crosses the link as YUV and is converted into the RGB frame
            ya, yb, xa, xb = even_rect(rect, H, W)
            self.engine.upload_yuv420_rect(self.frame_format, image, ya, yb, xa, xb, self._frame_pin, self._frame_stage, self._frame_dev)
        elif self._dev.type == "cuda":
            with torch.cuda.device(self._dev):
                rc = self.engine.lib.vt_upload_frame_rect(image.ctypes.data, H, W, ya, yb, xa, xb, self._frame_pin.data_ptr(),
                                                          self._frame_stage.data_ptr(), self._frame_dev.data_ptr(),
                                                          torch.cuda.current_stream(self._dev).cuda_stream)
            if rc != 0:
                raise RuntimeError(f"vt_upload_frame_rect failed ({rc})")
        else:
            a, b = ya * W * 3, yb * W * 3
            self._frame_dev[a:b].copy_(torch.from_numpy(image.reshape(-1)[a:b]))
        return H, W, crop_sz

    def _set_box(self, box, upload: bool = True):
        self._box_np[0, :] = [float(v) for v in box]
        if upload:
            self._box_dev.copy_(self._box_pin, non_blocking=True)

    # ------------------------------------------------------------------------------------------
    def initialize(self, image, info: dict):
        box = info['init_bbox']
        self._upload(image, box, self.params.template_factor)
        self._set_box(box)
        status = self.engine.tracks_init(self._frame_dev, self._off_dev, self._hw_dev, self._box_dev, first=0)
        # the reference keeps the uint8 template crop (vit_dist.py:55-57, self.z_patch_arr); the crop runs now (the frame buffer is
        # reused by the next frame), the device -> host copy only when the attribute is read
        self._z_patch_dev = self.engine.crop_normalize(self._frame_dev, self._off_dev, self._hw_dev, self._box_dev,
                                                       self.params.template_factor, self.params.template_size, want_u8=True)["u8"]
        self._z_patch_arr = None
        st = int(status.item())
        if st == 1:
            raise Exception('Too small bounding box.')
        if st != 0:
            raise ValueError("init_bbox crop lies outside the image (undefined behaviour in the reference)")
        self.state = info['init_bbox']
        self.frame_id = 0
        return None

    @property
    def z_patch_arr(self) -> np.ndarray:
        """uint8 [template_size, template_size, 3] template crop, as ``sample_target`` returned it (vit_dist.py:55-57)."""
        if self._z_patch_arr is None:
            if getattr(self, "_z_patch_dev", None) is None:
                raise AttributeError("z_patch_arr is set by initialize()")
            self._z_patch_arr = self._z_patch_dev[0].cpu().numpy()
        return self._z_patch_arr

    def track(self, image, info: dict = None):
        self.frame_id += 1
        H, W, crop_sz = self._upload(image, self.state, self.params.search_factor)
        resize_factor = self.params.search_size / crop_sz       # processing_utils.py:67
        self._set_box(self.state, upload=False)
        self._step_device()
        self._sync()
        # `confidence` is a 0-dim tensor on the model's device, as the reference's `score_map.max()` is (vit_dist.py:147-148); the
        # conversion is queued behind the step and never waited for
        confidence = self._out_dev[4].to(torch.float32)
        out = self._out_pin.tolist()
        if int(out[11]) == 1:
            raise Exception('Too small bounding box.')
        if int(out[11]) == 3:
            raise FloatingPointError("an activation left the fp16 operand range of the tensor-core path (or was non-finite): result "
                                     "withheld; construct the tracker with params.blocks_impl = 'simt' for these weights")
        if int(out[11]) != 0:
            raise ValueError("search crop lies outside the image (undefined behaviour in the reference)")
        pred_box = out[5:9]                                      # (cx, cy, w, h) as `.tolist()` of the fp32 tensor
        self.state = clip_box(self.map_box_back(pred_box, resize_factor), H, W, margin=10)
        self.last_detail = {"argmax": int(out[10]), "resize_factor": out[9], "window_max": out[12], "device_box": out[0:4]}
        return {"target_bbox": self.state, "confidence": confidence}

    def _step_device(self) -> None:
        """State upload + one tracking step + result download for the single track.  Every buffer involved is allocated once (frame
        buffer, pinned box, frame size, outputs, pinned result), so after the first frames the whole sequence - box H2D, the step's
        kernels, result D2H - is captured in a CUDA graph and replayed: one graph launch per frame (SURVEY 7.1 step 7).
        params.cuda_graph = False keeps plain launches."""
        def launch():
            self._box_dev.copy_(self._box_pin, non_blocking=True)
            self.engine.tracks_set_state(self._box_dev, first=0)
            self.engine.tracks_step(self._frame_dev, self._off_dev, self._hw_dev, first=0, n=1, out_boxes=self._out_boxes,
                                    out_detail=self._out_detail, update_state=False, detail=True)
            self._out_pin.copy_(self._out_dev, non_blocking=True)
        use_graph = self._dev.type == "cuda" and getattr(self.params, "cuda_graph", True)
        key = (self._hw, self._frame_dev.data_ptr() if self._frame_dev is not None else 0)
        if use_graph and getattr(self, "_graph_key", None) == key and self._graph is not None:
            self._graph.replay()
            return
        launch()
        if not use_graph or getattr(self, "_graph_failed", False):
            return
        # capture after a warm frame on these buffers (lazy one-off configuration inside the library has happened by then)
        self._graph_warm = getattr(self, "_graph_warm", 0) + 1 if getattr(self, "_graph_warm_key", None) == key else 1
        self._graph_warm_key = key
        if self._graph_warm < 2:
            return
        try:
            torch.cuda.current_stream(self._dev).synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                launch()
            self._graph, self._graph_key = g, key
        except Exception:
            self._graph, self._graph_key, self._graph_failed = None, None, True
            torch.cuda.synchronize(self._dev)

    def map_box_back(self, pred_box: list, resize_factor: float):
        """lib/test/tracker/vit_dist.py:150-156."""
        cx_prev, cy_prev = self.state[0] + 0.5 * self.state[2], self.state[1] + 0.5 * self.state[3]
        cx, cy, w, h = pred_box
        half_side = 0.5 * self.params.search_size / resize_factor
        cx_real = cx + (cx_prev - half_side)
        cy_real = cy + (cy_prev - half_side)
        return [cx_real - 0.5 * w, cy_real - 0.5 * h, w, h]


def get_tracker_class():
    return Vit_dist
