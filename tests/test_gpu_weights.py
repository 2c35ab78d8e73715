"""Weight ingestion through the C ABI (vt_set_tensor, vt_finalize_weights) on the tuned path (vit_48_h32) and the generic path.

Every name and shape the library accepts comes from one table per configuration: a complete state_dict loads with no unexpected
key; a key outside the table (an unknown name, or a block at index >= depth) comes back as unexpected, as
``load_state_dict(strict=False)`` would skip it; a tensor of another shape is refused.  Finalisation first checks that every
tensor of the table was set, and names the ones that were not.  Setting a tensor again on a finalised handle and finalising
again gives the bits of a fresh handle loaded with the changed weights.
"""
import ctypes

import pytest
import torch

from oracle import vt_oracle as O

VT_ERR_WEIGHTS = -3
# name: (C, heads, depth, head channels)
CONFIGS = {"vit_48_h32": (48, 1, 3, 32), "small": (96, 3, 2, 64)}


def _engine(name, n=2):
    from vittracker_b200 import load_cfg
    from vittracker_b200.engine import Engine
    C, heads, depth, hc = CONFIGS[name]
    cfg = load_cfg()
    cfg.MODEL.BACKBONE.CHANNELS, cfg.MODEL.BACKBONE.HEADS = C, heads
    cfg.MODEL.HEAD.NUM_CHANNELS = hc
    return Engine(cfg, max_tracks=n, depth=depth)


def _sd(name, seed=51):
    C, _, depth, hc = CONFIGS[name]
    return O.make_state_dict(seed=seed, stress=True, C=C, depth=depth, head_ch=hc)


def _crops(n=2, seed=52):
    g = torch.Generator().manual_seed(seed)
    return torch.randn((n, 3, 128, 128), generator=g), torch.randn((n, 3, 256, 256), generator=g)


def _forward_bits(e, z, x):
    out = e.forward(z, x, taps=True)
    torch.cuda.synchronize()
    return {k: v.cpu().contiguous().view(torch.int32) for k, v in out.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONFIGS))
def test_complete_state_dict_has_no_unexpected_keys(name):
    e = _engine(name)
    missing, unexpected = e.load_state_dict(_sd(name))
    assert missing == [] and unexpected == []


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONFIGS))
def test_unknown_key_and_block_past_depth_are_unexpected(name):
    C, _, depth, _ = CONFIGS[name]
    sd = _sd(name)
    sd["extra.weight"] = torch.ones(3)
    sd[f"blocks.{depth}.norm1.weight"] = torch.ones(C)
    e = _engine(name)
    _, unexpected = e.load_state_dict(sd)
    assert sorted(unexpected) == sorted(["extra.weight", f"blocks.{depth}.norm1.weight"])
    assert e.weights_loaded


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONFIGS))
def test_mis_shaped_tensor_is_refused(name):
    from vittracker_b200._lib import VtError
    sd = _sd(name)
    sd["blocks.0.attn.qkv.weight"] = sd["blocks.0.attn.qkv.weight"][:-1]
    with pytest.raises(VtError) as ei:
        _engine(name).load_state_dict(sd)
    assert ei.value.code == VT_ERR_WEIGHTS and "does not match expected" in str(ei.value)


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["patch_embed.net.2.bn.running_var", "blocks.1.attn.proj.bias", "box_head.conv2_offset.1.weight",
                                 "box_head.conv5_size.bias"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_missing_tensor_is_named(name, key):
    from vittracker_b200._lib import VtError
    sd = _sd(name)
    del sd[key]
    e = _engine(name)
    with pytest.raises(VtError) as ei:
        e.load_state_dict(sd)
    assert ei.value.code == VT_ERR_WEIGHTS and "missing tensors" in str(ei.value) and key in str(ei.value)
    assert not e.weights_loaded


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONFIGS))
def test_finalising_again_after_one_tensor_changes_matches_a_fresh_handle(name):
    key = "blocks.0.attn.qkv.weight"
    sd = _sd(name)
    z, x = _crops()
    e = _engine(name)
    e.load_state_dict(sd)
    before = _forward_bits(e, z, x)
    changed = dict(sd)
    changed[key] = sd[key] * 0.5
    a = changed[key].contiguous()
    shape = (ctypes.c_int64 * a.dim())(*a.shape)
    e._check(e.lib.vt_set_tensor(e.handle, key.encode(), ctypes.c_void_p(a.data_ptr()), shape, a.dim()))
    with torch.cuda.device(e.device):
        e._check(e.lib.vt_finalize_weights(e.handle, e._stream()))
    again = _forward_bits(e, z, x)
    fresh = _engine(name)
    fresh.load_state_dict(changed)
    want = _forward_bits(fresh, z, x)
    assert not torch.equal(before["score_map"], want["score_map"])
    for k in want:
        assert torch.equal(again[k], want[k]), k
