"""Model-side drop-in: ``build_ostrack_dist(cfg, depth=3, mode='eval')`` returning an object with
the reference model's inference surface (lib/models/vit_dist/vit_dist.py:57-155,159-198):
``forward(z=..., x=...)`` -> {'pred_boxes','score_map','size_map','offset_map'},
``box_head.cal_bbox(score, size_map, offset_map)``, ``load_state_dict(sd, strict=False)``,
``.cuda()`` / ``.eval()``.  All math runs in libvittrack_b200's sm_100a kernels."""
from __future__ import annotations

from typing import Dict, Optional

import torch

from .engine import Engine
from .weights import param_shapes, random_init_state_dict


class CenterHeadHandle:
    """Stands where ``network.box_head`` (CenterPredictor, lib/models/layers/head.py:98-201) stands:
    the tracker only reaches for ``cal_bbox`` and ``feat_sz``."""

    def __init__(self, model: "OstrackDistB200", feat_sz: int, stride: int):
        self._model = model
        self.feat_sz = feat_sz
        self.stride = stride
        self.img_sz = feat_sz * stride

    def cal_bbox(self, score_map_ctr, size_map, offset_map, return_score: bool = False):
        boxes = self._model.engine.cal_bbox(score_map_ctr, size_map, offset_map)
        if return_score:
            return boxes, score_map_ctr.flatten(1).max(dim=1, keepdim=True)[0]
        return boxes


class OstrackDistB200:
    def __init__(self, cfg, depth: int = 3, mode: str = "eval", blocks_impl: str = "tcgen05", max_tracks: int = 1,
                 chunk_tracks: int = 0, range_fallback: bool = False):
        if mode != "eval":
            raise NotImplementedError("only mode='eval' (inference) is implemented; the distillation/training "
                                      "branches of OstrackDist (vit_dist.py:69-73,97-119) are out of scope")
        self.cfg = cfg
        self.depth = depth
        self.mode = mode
        self.head_type = str(cfg.MODEL.HEAD.TYPE)
        self.feat_sz_s = int(cfg.TEST.SEARCH_SIZE) // int(cfg.MODEL.BACKBONE.STRIDE)
        self.feat_len_s = self.feat_sz_s ** 2
        self.box_head = CenterHeadHandle(self, self.feat_sz_s, int(cfg.MODEL.BACKBONE.STRIDE))
        self._blocks_impl = blocks_impl
        self._max_tracks = max_tracks
        self._chunk_tracks = chunk_tracks
        self._range_fallback = range_fallback            # tracking steps recompute range-flagged tracks on the fp32 kernels
        self._engine: Optional[Engine] = None
        self._device: Optional[int] = None
        self._sd: Dict[str, torch.Tensor] = random_init_state_dict(cfg, depth)
        self.training = False

    # -- nn.Module-like surface ----------------------------------------------------------------
    def load_state_dict(self, state_dict: Dict[str, torch.Tensor], strict: bool = True):
        known = param_shapes(self.cfg, self.depth)
        missing = [k for k in known if k not in state_dict]
        unexpected = [k for k in state_dict if k not in known]
        if strict and (missing or unexpected):
            raise RuntimeError(f"Error(s) in loading state_dict: missing {missing}, unexpected {unexpected}")
        for k, shape in known.items():
            if k in state_dict:
                t = state_dict[k].detach().cpu()
                if tuple(t.shape) != tuple(shape):
                    raise RuntimeError(f"size mismatch for {k}: {tuple(t.shape)} vs {tuple(shape)}")
                self._sd[k] = t.clone()
        if self._engine is not None:
            self._engine.load_state_dict(self._sd)
        return missing, unexpected

    def state_dict(self) -> Dict[str, torch.Tensor]:
        return dict(self._sd)

    def cuda(self, device=None):
        self._device = torch.cuda.current_device() if device is None else torch.device(device).index if not isinstance(device, int) else device
        _ = self.engine
        return self

    def to(self, device):
        return self.cuda(device)

    def eval(self):
        return self

    @property
    def engine(self) -> Engine:
        if self._engine is None:
            self._engine = Engine(self.cfg, max_tracks=self._max_tracks, chunk_tracks=self._chunk_tracks,
                                  device=self._device, blocks_impl=self._blocks_impl, depth=self.depth)
            self._engine.load_state_dict(self._sd)
            if self._range_fallback:
                self._engine.set_range_fallback(True)
        return self._engine

    # -- inference -----------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, z: torch.Tensor, x: torch.Tensor, return_taps: bool = False):
        return self.engine.forward(z, x, taps=return_taps)

    __call__ = forward


def build_ostrack_dist(cfg, depth: int = 3, mode: str = "eval", **kw) -> OstrackDistB200:
    """Same signature as the reference builder (vit_dist.py:159); eval mode only."""
    return OstrackDistB200(cfg, depth=depth, mode=mode, **kw)
