"""vittracker_b200: B200-native (sm_100a) implementation of VitTracker's per-frame inference hot path
(tracker ``vit_dist``, experiment ``vit_48_h32_noKD``) behind the reference's own tracker / model API.

Python here is host-side plumbing (device memory, streams, torch.distributed); every computation is
a call through the C ABI of ``lib/libvittrack_b200.so`` (include/vittrack_b200.h) into hand-written
CUDA kernels.  There is no CPU fallback."""
from .config import cfg, load_cfg, update_config_from_file  # noqa: F401
from .params import TrackerParams, parameters  # noqa: F401


def __getattr__(name):
    # torch-dependent pieces are imported lazily so that `import vittracker_b200` stays cheap
    if name in ("Engine", "hann2d_window"):
        from . import engine
        return getattr(engine, name)
    if name in ("build_ostrack_dist", "OstrackDistB200"):
        from . import model
        return getattr(model, name)
    if name in ("Vit_dist", "get_tracker_class", "BaseTracker", "clip_box"):
        from . import tracker
        return getattr(tracker, name)
    if name in ("BatchedTracker", "ShardedTracker", "FramePool", "PipelinedFrameFeeder", "YuvSurfaces", "shard_range"):
        from . import batched
        return getattr(batched, name)
    if name in ("Sequence", "MultiSequenceRunner", "BatchedBackend", "run_sequences", "save_tracker_output", "read_image"):
        from . import sequences
        return getattr(sequences, name)
    if name in ("TrackRecords",):
        from . import records
        return getattr(records, name)
    if name in ("CropPreprocessor", "NestedTensor"):
        from . import preprocess
        return getattr(preprocess, name)
    raise AttributeError(name)
