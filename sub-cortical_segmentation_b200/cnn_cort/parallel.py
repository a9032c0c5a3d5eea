"""Multi-GPU sharding of the hot path (one process per GPU, torch.distributed for the plumbing).

Inference is embarrassingly parallel (every voxel depends only on the read-only volume, atlas and
weights), so it shards with NO collective: by volume (`shard_items`) or, inside one volume, by
contiguous x-slabs of the candidate box (`shard_box`) -- a slab is a contiguous range of the
C-ordered candidate list the reference iterates over (base.py:379-382).  Training is data-parallel:
the only exchange is one all-reduce of the flat 883 455-float gradient buffer per step
(`allreduce_gradients`), after which every rank applies the same Adam step.
"""
import os


def dist_info():
    """(rank, world, local_rank) from torch.distributed if initialised, else from the torchrun env."""
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size(), int(os.environ.get("LOCAL_RANK", dist.get_rank()))
    except ImportError:
        pass
    return int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))


def shard_range(n, rank, world):
    """Contiguous [start, stop) share of n items; sizes differ by at most one, ranks in order."""
    base, extra = divmod(int(n), int(world))
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def shard_items(items, rank, world):
    """Round-robin share of a list of volumes / scan paths (BASELINE config 3: 64 volumes over N GPUs)."""
    return list(items[rank::world])


def shard_box(box, rank, world):
    """Split a half-open candidate box (x0,x1,y0,y1,z0,z1) into x-slabs; None if this rank gets nothing."""
    x0, x1 = int(box[0]), int(box[1])
    a, b = shard_range(x1 - x0, rank, world)
    if a == b:
        return None
    return (x0 + a, x0 + b) + tuple(int(v) for v in box[2:])


def shard_batch(indices, rank, world):
    """This rank's samples of one global minibatch (strided so that class order does not matter)."""
    return indices[rank::world]


def dataset_fingerprint(xs, y):
    """int64 [4]: size, CRC of the labels, CRCs of a strided sample of the first and last input array"""
    import zlib
    import numpy as np
    n = len(y)
    step = max(1, n // 64)
    return np.array([n, zlib.crc32(np.ascontiguousarray(y).tobytes()),
                     zlib.crc32(np.ascontiguousarray(xs[0][::step]).tobytes()),
                     zlib.crc32(np.ascontiguousarray(xs[-1][::step]).tobytes())], dtype=np.int64)


def scan_set_fingerprint(samples, atlas_rows, labels, volumes):
    """int64 [5] of a ScanTrainingSet: size, CRCs of the sample table, the labels and the atlas rows, and one CRC over the
    shape and a strided sample (about 4096 voxels) of every volume (CUDA tensors)"""
    import zlib
    import numpy as np
    crc = 0
    for v in volumes:
        flat = v.reshape(-1)
        crc = zlib.crc32(np.asarray(tuple(v.shape), np.int64).tobytes(), crc)
        crc = zlib.crc32(flat[::max(1, flat.numel() // 4096)].cpu().numpy().tobytes(), crc)
    return np.array([len(labels), zlib.crc32(np.ascontiguousarray(samples).tobytes()), zlib.crc32(np.ascontiguousarray(labels).tobytes()),
                     zlib.crc32(np.ascontiguousarray(atlas_rows).tobytes()), crc], dtype=np.int64)


def assert_same_dataset(xs, y, device=None):
    """Data-parallel fit shards every global minibatch by position, so all ranks must hold the same arrays in the same
    order.  Compares a fingerprint with rank 0's and raises on every rank if any rank differs."""
    assert_same_fingerprint(dataset_fingerprint(xs, y), device)


def assert_same_fingerprint(fingerprint, device=None):
    """Raises on every rank unless every rank's int64 fingerprint equals rank 0's."""
    import torch
    import torch.distributed as dist
    mine = torch.from_numpy(fingerprint)
    if device is not None and dist.get_backend() == "nccl":
        mine = mine.to(device)
    ref = mine.clone()
    dist.broadcast(ref, 0)
    bad = (ref != mine).any().to(torch.int64).reshape(1)
    dist.all_reduce(bad, op=dist.ReduceOp.MAX)
    if int(bad.item()):
        raise ValueError("data-parallel fit: the ranks hold different training sets (size / order / content); build the set "
                         "once (a fixed seed for load_data's negative sampling and generate_training_set) or broadcast it")


def allreduce_gradients(grads, loss=None):
    """Sum-all-reduce the flat gradient buffer (and the scalar loss) in place.  The kernels already divide
    by the GLOBAL batch size, so the sum is the global-batch gradient; the BN-statistics slots carry
    per-rank batch statistics whose sum sc_adam_step divides by the world size (stat_scale)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return 1
    dist.all_reduce(grads)
    if loss is not None:
        dist.all_reduce(loss)
    return dist.get_world_size()


def segment_volume_sharded(ctx, vol, atlas, box=None, cand_mask=None, label_vol=None, proba_vol=None):
    """Each rank segments its x-slab of the box into its own (full-size) output volumes: disjoint
    voxel sets, no collective.  Returns the slab this rank wrote (or None)."""
    rank, world, _ = dist_info()
    if box is None:
        box = (0, vol.shape[0], 0, vol.shape[1], 0, vol.shape[2])
    mine = shard_box(box, rank, world)
    if mine is not None:
        ctx.segment_volume(vol, atlas, box=mine, cand_mask=cand_mask, label_vol=label_vol, proba_vol=proba_vol)
    return mine
