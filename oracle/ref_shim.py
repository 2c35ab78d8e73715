"""Import shim that lets the UNMODIFIED reference modules of the original project run on CPU (TEST INFRASTRUCTURE; used only by
oracle/make_golden.py and, where a checkout of the original is present, by tests that re-pin the oracle against it.  Never imported
by the product).  The checkout is looked for at oracle/_ref (kept out of git) unless $VT_REFERENCE_ROOT names another place.

The reference imports packages this image lacks (SURVEY.md 8c): timm, easydict, visdom, lmdb,
jpeg4py, matplotlib, torch._six; hard-codes ``.cuda()`` (lib/test/tracker/vit_dist.py:27,34,
lib/test/tracker/data_utils.py:8-16) and machine paths (lib/test/evaluation/local.py).  The shim
installs minimal stand-ins in ``sys.modules`` BEFORE the reference is imported and turns ``.cuda()``
into identity.  The only arithmetic it supplies is timm's ``Block``/``Attention``/``Mlp`` -
restated from timm's published vision_transformer.py as the reference's authors copied it at
tracking/onnxexport.py:126-225 (non-fused branch: q*scale, softmax, @v; scale = head_dim**-0.5).
"""
from __future__ import annotations

import os
import sys
import types

import torch
import torch.nn as nn

REFERENCE_ROOT = os.environ.get("VT_REFERENCE_ROOT") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "lib", "test", "tracker", "vit_dist.py"))


# --- timm stand-in ---------------------------------------------------------------------------
class Mlp(nn.Module):
    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0., **kw):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = act_layer()
        self.fc2 = nn.Linear(hidden_features, out_features)

    def forward(self, x):
        return self.fc2(self.act(self.fc1(x)))


class Attention(nn.Module):
    def __init__(self, dim, num_heads=8, qkv_bias=False, qk_norm=False, attn_drop=0., proj_drop=0., **kw):
        super().__init__()
        self.num_heads = num_heads
        self.head_dim = dim // num_heads
        self.scale = self.head_dim ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.proj = nn.Linear(dim, dim)

    def forward(self, x):
        B, N, C = x.shape
        qkv = self.qkv(x).reshape(B, N, 3, self.num_heads, self.head_dim).permute(2, 0, 3, 1, 4)
        q, k, v = qkv.unbind(0)
        q = q * self.scale
        attn = (q @ k.transpose(-2, -1)).softmax(dim=-1)
        x = (attn @ v).transpose(1, 2).reshape(B, N, C)
        return self.proj(x)


class Block(nn.Module):
    def __init__(self, dim, num_heads, mlp_ratio=4., qkv_bias=False, **kw):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim)
        self.attn = Attention(dim, num_heads=num_heads, qkv_bias=qkv_bias)
        self.norm2 = nn.LayerNorm(dim)
        self.mlp = Mlp(in_features=dim, hidden_features=int(dim * mlp_ratio))

    def forward(self, x):
        x = x + self.attn(self.norm1(x))
        x = x + self.mlp(self.norm2(x))
        return x


class _Identityish(nn.Module):
    def __init__(self, *a, **k):
        super().__init__()

    def forward(self, x, *a, **k):
        return x


def _to_2tuple(x):
    return tuple(x) if isinstance(x, (tuple, list)) else (x, x)


class _EasyDict(dict):
    """Minimal easydict.EasyDict: attribute access, nested dicts converted recursively."""

    def __init__(self, d=None, **kw):
        super().__init__()
        d = dict(d or {}, **kw)
        for k, v in d.items():
            setattr(self, k, v)

    def __setattr__(self, k, v):
        if isinstance(v, dict) and not isinstance(v, _EasyDict):
            v = _EasyDict(v)
        elif isinstance(v, (list, tuple)):
            v = type(v)(_EasyDict(x) if isinstance(x, dict) and not isinstance(x, _EasyDict) else x for x in v)
        super().__setitem__(k, v)
        super().__setattr__(k, v)

    __setitem__ = __setattr__


def _module(name: str, **attrs) -> types.ModuleType:
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    m.__path__ = []          # behave as a package so sub-imports resolve through sys.modules
    sys.modules[name] = m
    return m


class _Anything:
    """Stand-in object: any attribute / call yields another stand-in (visdom, matplotlib ...)."""

    def __init__(self, *a, **k):
        pass

    def __getattr__(self, n):
        return _Anything()

    def __call__(self, *a, **k):
        return _Anything()


class _AnyModule(types.ModuleType):
    def __getattr__(self, n):
        if n.startswith("__"):
            raise AttributeError(n)
        return _Anything


_installed = False


def install() -> None:
    """Install the stand-ins and put the reference on sys.path (idempotent)."""
    global _installed
    if _installed:
        return
    if not available():
        raise RuntimeError(f"no checkout of the original project at {REFERENCE_ROOT} (set VT_REFERENCE_ROOT to use another)")

    vt = dict(Block=Block, Attention=Attention, Mlp=Mlp, LayerScale=_Identityish, DropPath=_Identityish,
              PatchEmbed=_Identityish, Final=object, use_fused_attn=lambda *a, **k: False,
              _cfg=lambda *a, **k: {}, VisionTransformer=nn.Module, _load_weights=lambda *a, **k: None,
              trunc_normal_=nn.init.trunc_normal_, lecun_normal_=lambda t: t, named_apply=lambda *a, **k: None,
              _init_vit_weights=lambda *a, **k: None, HybridEmbed=_Identityish, resize_pos_embed=lambda *a, **k: None)
    layers = dict(Mlp=Mlp, DropPath=_Identityish, trunc_normal_=nn.init.trunc_normal_,
                  lecun_normal_=lambda t: t, to_2tuple=_to_2tuple, PatchEmbed=_Identityish)
    timm = _module("timm")
    timm.models = _module("timm.models")
    timm.models.vision_transformer = _module("timm.models.vision_transformer", **vt)
    timm.models.layers = _module("timm.models.layers", **layers)
    timm.layers = _module("timm.layers", **layers)
    timm.models.helpers = _module("timm.models.helpers", build_model_with_cfg=lambda *a, **k: None,
                                  named_apply=lambda *a, **k: None, adapt_input_conv=lambda *a, **k: None,
                                  checkpoint_seq=lambda *a, **k: None)
    timm.models.registry = _module("timm.models.registry", register_model=lambda f: f)
    timm.data = _module("timm.data", IMAGENET_DEFAULT_MEAN=(0.485, 0.456, 0.406),
                        IMAGENET_DEFAULT_STD=(0.229, 0.224, 0.225), IMAGENET_INCEPTION_MEAN=(0.5,) * 3,
                        IMAGENET_INCEPTION_STD=(0.5,) * 3)

    _module("easydict", EasyDict=_EasyDict)
    for name in ("visdom", "visdom.server", "lmdb", "jpeg4py", "matplotlib", "matplotlib.pyplot", "matplotlib.patches",
                 "matplotlib.colors", "tikzplotlib", "pycocotools", "pycocotools.coco", "thop", "wandb",
                 "tensorboardX", "segment_anything"):
        if name not in sys.modules:
            try:
                __import__(name)
            except Exception:
                sys.modules[name] = _AnyModule(name)
                sys.modules[name].__path__ = []
    if "torch._six" not in sys.modules:
        _module("torch._six", string_classes=(str, bytes), int_classes=(int,), container_abcs=__import__("collections").abc)
        torch._six = sys.modules["torch._six"]

    # .cuda() -> identity: the reference runs on the CPU here
    torch.Tensor.cuda = lambda self, *a, **k: self
    nn.Module.cuda = lambda self, *a, **k: self

    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    _installed = True


def load_reference():
    """Import the reference's hot-path modules; returns a namespace of the objects tests need."""
    install()
    import importlib
    ns = types.SimpleNamespace()
    ns.processing_utils = importlib.import_module("lib.train.data.processing_utils")
    ns.sample_target = ns.processing_utils.sample_target
    ns.hann = importlib.import_module("lib.test.utils.hann")
    ns.box_ops = importlib.import_module("lib.utils.box_ops")
    ns.vit_dist_model = importlib.import_module("lib.models.vit_dist.vit_dist")
    ns.build_ostrack_dist = ns.vit_dist_model.build_ostrack_dist
    ns.config = importlib.import_module("lib.config.vit_dist.config")
    ns.data_utils = importlib.import_module("lib.test.tracker.data_utils")
    ns.tracker_mod = importlib.import_module("lib.test.tracker.vit_dist")
    ns.Vit_dist = ns.tracker_mod.get_tracker_class()
    ns.yaml = os.path.join(REFERENCE_ROOT, "experiments", "vit_dist", "vit_48_h32_noKD.yaml")
    return ns


def reference_cfg():
    ns = load_reference()
    ns.config.update_config_from_file(ns.yaml)
    return ns.config.cfg


def build_reference_tracker(state_dict, tmpdir: str):
    """Vit_dist(params, dataset_name) from the reference, fed a checkpoint holding ``state_dict``."""
    ns = load_reference()
    cfg = reference_cfg()
    ckpt = os.path.join(tmpdir, "OstrackDist_ep0300.pth.tar")
    torch.save({"net": state_dict}, ckpt)

    class Params:       # the attribute bag lib/test/parameter/vit_dist.py:7-30 builds
        pass

    p = Params()
    p.cfg = cfg
    p.template_factor, p.template_size = cfg.TEST.TEMPLATE_FACTOR, cfg.TEST.TEMPLATE_SIZE
    p.search_factor, p.search_size = cfg.TEST.SEARCH_FACTOR, cfg.TEST.SEARCH_SIZE
    p.checkpoint = ckpt
    p.save_all_boxes = False
    p.debug = 0
    return ns.Vit_dist(p, "synthetic")
