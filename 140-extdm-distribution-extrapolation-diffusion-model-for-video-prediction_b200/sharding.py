"""Multi-GPU: videos are independent units (SURVEY.md section 8e) -- each rank runs the full sampler on its slice,
no collective on the data path; one all-gather of the predicted frames at the end.

Seeded sampling keys each video's noise by a seed derived from its *global* index (video_seeds), so a video is sampled
with the same noise whichever rank, batch or GPU count it lands on."""
import numpy as np
import torch
import torch.distributed as dist

_M64 = (1 << 64) - 1


def _u64(v):
    """int, sequence of ints or integer tensor -> 1-D uint64 array of the values mod 2**64."""
    if torch.is_tensor(v):
        return v.detach().cpu().reshape(-1).to(torch.int64).numpy().astype(np.uint64)
    return np.array([int(x) & _M64 for x in np.atleast_1d(np.asarray(v, dtype=object))], dtype=np.uint64)


def _splitmix64(x):
    """The output function of splitmix64 (Steele, Lea and Flood, OOPSLA 2014) applied to x + 0x9E3779B97F4A7C15."""
    with np.errstate(over="ignore"):
        z = x + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def video_seeds(base_seed, video_ids, round=0):
    """Sampler seeds (int64 tensor, values in [0, 2**62)) of the given *global* video indices at rollout round
    `round`.  base_seed and video_ids are each one int or one value per video (then of equal length); the result has
    one seed per video.  With every value taken mod 2**64 and m = _splitmix64:

        seed = m(m(m(base_seed) ^ video_id) ^ round) >> 2

    A pure host function: the seed of a video depends on (base_seed, video_id, round) only, not on the batch, the
    rank or the number of ranks it is sampled on."""
    ids = _u64(video_ids)
    base = _u64(base_seed)
    if base.size != 1 and ids.size != 1 and base.size != ids.size:
        raise ValueError(f"video_seeds: {base.size} base seeds for {ids.size} videos")
    h = _splitmix64(_splitmix64(_splitmix64(base) ^ ids) ^ _u64(round))
    return torch.from_numpy((h >> np.uint64(2)).astype(np.int64))


def shard_range(n_videos, rank, world):
    """Contiguous, balanced slice [lo, hi) of the video indices for `rank` (first ranks take the remainder)."""
    base, rem = divmod(n_videos, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def gather_predictions(local, n_videos):
    """All-gather per-rank predictions (b_r, 3, T, H, W) into (n_videos, 3, T, H, W) in rank order.
    Ragged shards are padded to the largest shard for the collective and trimmed afterwards."""
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return local
    world, rank = dist.get_world_size(), dist.get_rank()
    sizes = [shard_range(n_videos, r, world) for r in range(world)]
    mx = max(hi - lo for lo, hi in sizes)
    pad = torch.zeros(mx, *local.shape[1:], dtype=local.dtype, device=local.device)
    pad[: local.shape[0]] = local
    out = torch.empty(world * mx, *local.shape[1:], dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, pad)
    return torch.cat([out[r * mx: r * mx + (hi - lo)] for r, (lo, hi) in enumerate(sizes)], dim=0)
