"""The argument checks every C-ABI entry point and Engine method makes before any launch: for each entry point that takes n, first
or slots, every kind of bad argument gets its status code and a message and launches nothing, an empty batch with null pointers is a
no-op, and every Engine method refuses a tensor of the wrong dtype, device or shape, or a non-contiguous one, with ValueError."""
import numpy as np
import pytest
import torch

from oracle import vt_oracle as O

pytestmark = pytest.mark.gpu
M = 8                                   # max_tracks
LAST = (2, 3)                           # the fixture's last step: tracks [2, 5)
INT_MAX = 2 ** 31 - 1
INVALID, STATE = -1, -4
H = W = 64

# argument markers of the table: a required pointer, an optional one, slots, records, first, n
P, O_, S, R, F, N = (object() for _ in range(6))
POINTERS = (P, O_, S, R)

# entry point -> (arguments after the handle and before the stream, what its n indexes: a batch of items, tracks of the handle, a
# slot list, or tracks of the last step)
ENTRIES = {
    "vt_crop_normalize": ((P, P, P, P, 2.0, 128, N, P, O_, O_, O_, O_), "batch"),
    "vt_forward": ((P, P, N, O_, O_, O_, O_, O_), "batch"),
    "vt_cal_bbox": ((P, P, P, N, P), "batch"),
    "vt_tracks_init": ((P, P, P, P, F, N, O_), "range"),
    "vt_tracks_init_slots": ((P, P, P, P, S, N, O_), "list"),
    "vt_tracks_step": ((P, P, P, F, N, P, O_, 0), "range"),
    "vt_tracks_step_slots": ((P, P, P, S, N, P, O_, 0), "list"),
    "vt_tracks_export": ((F, N, R), "range"),
    "vt_tracks_export_slots": ((S, N, R, O_), "list"),
    "vt_tracks_import": ((R, F, N, O_), "range"),
    "vt_tracks_import_slots": ((R, S, N, O_), "list"),
    "vt_tracks_get_state": ((P, F, N), "range"),
    "vt_tracks_set_state": ((P, F, N), "range"),
    "vt_tracks_last_maps": ((F, N, O_, O_, O_), "last"),
    "vt_yuv420_to_rgb": ((1, P, P, P, P, P, N), "batch"),
    "vt_yuv420_crop_to_rgb": ((1, P, P, P, O_, 2.0, F, N, P, P), "batch"),
}
# vt_yuv420_crop_to_rgb without boxes crops around the state of tracks [first, first + n)
STATE_CROP = ((1, P, P, P, None, 4.0, F, N, P, P), "range")


def _args(spec, first, n, addr, null=None, records=None):
    """The arguments of one call: every pointer `addr` (None for an empty batch), except position `null` and a misaligned `records`."""
    out = []
    for i, a in enumerate(spec):
        if a is F:
            out.append(first)
        elif a is N:
            out.append(n)
        elif any(a is p for p in POINTERS):
            out.append(None if i == null or addr is None else records if a is R and records is not None else addr)
        else:
            out.append(a)
    return out


def _bad_calls(spec, kind, addr):
    """(first of its n == 0 call, [(label, arguments, status) of every refused call]) of one entry point."""
    lo, count = LAST if kind == "last" else (0, M)
    code = STATE if kind == "last" else INVALID
    ranges = [("n < 0", lo, -1, code)]
    if kind == "list":
        ranges.append(("n > max_tracks", 0, M + 1, INVALID))
    if kind in ("range", "last"):
        ranges += [("first < 0" if kind == "range" else "first before the last step", lo - 1, 1, code),
                   ("first + n one past the end", lo + 1, count, code), ("first = INT_MAX, n = 1", INT_MAX, 1, code)]
    calls = [(label, _args(spec, first, n, addr), status) for label, first, n, status in ranges]
    for i, a in enumerate(spec):
        if any(a is p for p in (P, S, R)):
            calls.append((f"null argument {i}", _args(spec, lo, 1, addr, null=i), INVALID))
        if a is R:
            calls.append(("misaligned records", _args(spec, lo, 1, addr, records=addr + 1), INVALID))
    return lo, calls


@pytest.fixture(scope="module")
def engine():
    from vittracker_b200 import load_cfg
    from vittracker_b200.engine import Engine
    e = Engine(load_cfg(), max_tracks=M)
    e.load_state_dict(O.make_state_dict(seed=5, stress=True))
    dev = e.device
    frames = torch.from_numpy(O.synth_frames(1, H, W, seed=3)).to(dev).reshape(-1)
    boxes = torch.tensor([[20.0, 22.0, 14.0, 12.0]] * M, dtype=torch.float64, device=dev)
    e.tracks_init(frames, torch.zeros(M, dtype=torch.int64, device=dev), _hw(M, dev), boxes)
    e.frames = frames
    return e


def _hw(n, dev):
    return torch.tensor([[H, W]] * n, dtype=torch.int32, device=dev)


def test_bad_arguments_are_refused_before_any_launch(engine):
    lib, h, dev = engine.lib, engine.handle, engine.device
    lo, n = LAST
    engine.tracks_step(engine.frames, torch.zeros(n, dtype=torch.int64, device=dev), _hw(n, dev), first=lo, n=n)
    buf = torch.zeros(1 << 20, dtype=torch.uint8, device=dev)                      # every pointer of a refused call; never read
    addr = buf.data_ptr()
    torch.cuda.synchronize(dev)
    before = engine.launch_count
    tables = [(name, *ENTRIES[name]) for name in ENTRIES] + [("vt_yuv420_crop_to_rgb (state)", *STATE_CROP)]
    for name, spec, kind in tables:
        entry = name.split()[0]
        fn = getattr(lib, entry)
        lo, calls = _bad_calls(spec, kind, addr)
        assert fn(None, *_args(spec, lo, 1, addr), None) == INVALID, (name, "null handle")
        for label, args, status in calls:
            assert lib.vt_weights_fingerprint(h, None) == INVALID                  # leaves a message of its own
            assert fn(h, *args, None) == status, (name, label)
            assert lib.vt_last_error(h).startswith(entry.encode() + b": "), (name, label, lib.vt_last_error(h))
            assert engine.launch_count == before, (name, label)
        assert fn(h, *_args(spec, lo, 0, None), None) == 0, (name, "n == 0 with null pointers")
    assert engine.launch_count == before


def _mutations(t, shaped):
    """Wrong dtype, wrong device, one entry short in the last dimension (arrays whose shape is read), and the same values at a
    non-contiguous stride."""
    other = {torch.uint8: torch.int8, torch.int64: torch.int32, torch.int32: torch.int64, torch.float64: torch.float32,
             torch.float32: torch.float64}[t.dtype]
    out = {"dtype": t.to(other), "device": t.to("cuda" if t.device.type == "cpu" else "cpu")}
    if shaped:
        out["shape"] = t[..., :-1]
    if t.numel() > 1:
        out["non-contiguous"] = torch.stack([t, t], -1)[..., 0]
    return out


def test_engine_methods_refuse_bad_tensors_before_any_launch(engine):
    e, dev, n = engine, engine.device, 2
    frames = torch.from_numpy(O.synth_frames(1, H, W, seed=4)).to(dev).reshape(-1)
    off, hw = torch.zeros(n, dtype=torch.int64, device=dev), _hw(n, dev)
    boxes = torch.tensor([[20.0, 22.0, 14.0, 12.0]] * n, dtype=torch.float64, device=dev)
    slots = torch.tensor([6, 7], dtype=torch.int32, device=dev)
    out_boxes, out_detail = torch.zeros((n, 5), dtype=torch.float64, device=dev), torch.zeros((n, 8), dtype=torch.float64, device=dev)
    records = e.tracks_export(0, n)
    yuv = torch.full((H * 3 // 2 * W,), 128, dtype=torch.uint8, device=dev)
    rgb = torch.zeros(((n + 1) * H * W * 3,), dtype=torch.uint8, device=dev)
    rgb_off = torch.arange(n, dtype=torch.int64, device=dev) * (H * W * 3)
    planes = torch.tensor([[yuv.data_ptr(), yuv.data_ptr() + H * W, 0]] * n, dtype=torch.int64, device=dev)
    pitches = torch.tensor([[W, W]] * n, dtype=torch.int32, device=dev)
    staging = torch.zeros(H * W * 3 // 2, dtype=torch.uint8).pin_memory()
    staging_dev = torch.zeros(H * W * 3 // 2, dtype=torch.uint8, device=dev)
    image = np.full((H * 3 // 2, W), 128, np.uint8)
    counter = torch.zeros(1, dtype=torch.int64, device=dev)
    z, x = torch.zeros((n, 3, 128, 128), device=dev), torch.zeros((n, 3, 256, 256), device=dev)
    maps = [torch.zeros((n, c, 16, 16), device=dev) for c in (1, 2, 2)]
    # method -> (call over a dict of its tensors, the tensors, the names whose shape is read; forward and cal_bbox convert dtype,
    # device and layout as the reference model's callers expect, so only their shapes can be wrong)
    calls = {
        "crop_normalize": (lambda a: e.crop_normalize(a["frames"], a["off"], a["hw"], a["boxes"], 2.0, 128),
                           {"frames": frames, "off": off, "hw": hw, "boxes": boxes}, ("off", "hw", "boxes")),
        "forward": (lambda a: e.forward(a["z"], a["x"]), {"z": z, "x": x}, ("z", "x")),
        "cal_bbox": (lambda a: e.cal_bbox(a["score"], a["size"], a["offset"]),
                     {"score": maps[0], "size": maps[1], "offset": maps[2]}, ("score", "size", "offset")),
        "yuv420_to_rgb": (lambda a: e.yuv420_to_rgb(a["src"], a["src_off"], a["hw"], a["dst"], a["dst_off"], "nv12"),
                          {"src": yuv, "src_off": torch.zeros(n, dtype=torch.int64, device=dev), "hw": hw, "dst": rgb, "dst_off": rgb_off},
                          ("src_off", "hw", "dst_off")),
        "upload_yuv420_rect": (lambda a: e.upload_yuv420_rect("nv12", image, 0, 8, 0, 8, a["staging"], a["staging_dev"], a["frame"]),
                               {"staging": staging, "staging_dev": staging_dev, "frame": rgb}, ()),
        "yuv420_crop_to_rgb": (lambda a: e.yuv420_crop_to_rgb("nv12", a["planes"], a["pitches"], a["hw"], a["dst"], a["dst_off"], 2.0,
                                                              boxes=a["boxes"]),
                               {"planes": planes, "pitches": pitches, "hw": hw, "dst": rgb, "dst_off": rgb_off, "boxes": boxes},
                               ("planes", "pitches", "hw", "dst_off", "boxes")),
        "tracks_init": (lambda a: e.tracks_init(a["frames"], a["off"], a["hw"], a["boxes"], first=6),
                        {"frames": frames, "off": off, "hw": hw, "boxes": boxes}, ("off", "hw", "boxes")),
        "tracks_step": (lambda a: e.tracks_step(a["frames"], a["off"], a["hw"], first=6, n=n, out_boxes=a["out"], out_detail=a["detail"]),
                        {"frames": frames, "off": off, "hw": hw, "out": out_boxes, "detail": out_detail}, ("off", "hw", "out", "detail")),
        "tracks_init_slots": (lambda a: e.tracks_init_slots(a["frames"], a["off"], a["hw"], a["boxes"], a["slots"]),
                              {"frames": frames, "off": off, "hw": hw, "boxes": boxes, "slots": slots}, ("off", "hw", "boxes", "slots")),
        "tracks_step_slots": (lambda a: e.tracks_step_slots(a["frames"], a["off"], a["hw"], a["slots"], a["out"], a["detail"]),
                              {"frames": frames, "off": off, "hw": hw, "slots": slots, "out": out_boxes, "detail": out_detail},
                              ("off", "hw", "slots", "out", "detail")),
        "set_range_fallback": (lambda a: e.set_range_fallback(False, a["counter"]), {"counter": counter}, ("counter",)),
        "tracks_export": (lambda a: e.tracks_export(6, n, out=a["out"]), {"out": records.clone()}, ("out",)),
        "tracks_export_slots": (lambda a: e.tracks_export_slots(a["slots"], out=a["out"]), {"slots": slots, "out": records.clone()},
                                ("slots", "out")),
        "tracks_import": (lambda a: e.tracks_import(a["records"], first=6), {"records": records}, ("records",)),
        "tracks_import_slots": (lambda a: e.tracks_import_slots(a["records"], a["slots"]), {"records": records, "slots": slots},
                                ("records", "slots")),
        "tracks_set_state": (lambda a: e.tracks_set_state(a["boxes"], first=6), {"boxes": boxes}, ("boxes",)),
    }
    for name, (call, tensors, shaped) in calls.items():
        call(tensors)                                                               # the unaltered call is accepted
    torch.cuda.synchronize(dev)
    before = e.launch_count
    for name, (call, tensors, shaped) in calls.items():
        for arg, t in tensors.items():
            converted = name in ("forward", "cal_bbox")
            for what, bad in _mutations(t, arg in shaped).items():
                if converted and what != "shape":
                    continue
                with pytest.raises(ValueError):
                    call({**tensors, arg: bad})
        if "records" in tensors or "out" in tensors and tensors["out"].dtype == torch.uint8:
            arg = "records" if "records" in tensors else "out"
            shifted = torch.zeros(records.numel() + 16, dtype=torch.uint8, device=dev)[1:1 + records.numel()].view(records.shape)
            with pytest.raises(ValueError):
                call({**tensors, arg: shifted})                                     # misaligned records
    assert e.launch_count == before
