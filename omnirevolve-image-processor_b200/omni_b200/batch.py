"""Frame batches over several GPUs: the path shards by frame with NO data-path collective (SURVEY 8e).

One process per GPU (torchrun).  Each rank takes a contiguous block of ceil(B/G) frames, runs them through the pipelined
host call on its own device (groups of 32 / K frames per device pass), keeps its packed masks/edges in its own (pinned)
host buffers, and only the per-frame counts (the numbers the reference logs: pixels, mask_nonzero, edge nz) are gathered
to rank 0 in frame order.  bench.py's `configs3` record and tests/test_gpu_packed.py run exactly this.
torch.distributed is plumbing here: gloo on CPU boxes (tests), nccl on GPU boxes.
"""
from __future__ import annotations

import numpy as np


def shard_range(n_frames: int, world: int, rank: int) -> range:
    """Contiguous block of ceil(B/G) frames for `rank` (the last ranks may get fewer or none)."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("bad world/rank")
    per = -(-n_frames // world) if n_frames > 0 else 0
    lo = min(n_frames, rank * per)
    return range(lo, min(n_frames, lo + per))


def run_shard(frames, frame_ids, compute):
    """compute(frame) -> int64 array [K,3] of counts; returns {frame_id: counts} for this rank's frames."""
    return {int(i): np.asarray(compute(f), dtype=np.int64) for i, f in zip(frame_ids, frames)}


def gather_counts(local: dict, n_frames: int, K: int, dist=None) -> np.ndarray | None:
    """All ranks' {frame_id: counts[K,3]} -> on rank 0 one int64 array [n_frames, K, 3] in frame order."""
    if dist is None or not dist.is_initialized() or dist.get_world_size() == 1:
        parts = [local]
        rank = 0
    else:
        rank = dist.get_rank()
        parts = [None] * dist.get_world_size() if rank == 0 else None
        dist.gather_object(local, parts, dst=0)
    if rank != 0:
        return None
    out = np.full((n_frames, K, 3), -1, np.int64)
    for part in parts:
        for i, c in part.items():
            if not (0 <= i < n_frames) or out[i, 0, 0] != -1:
                raise RuntimeError(f"frame {i} reported twice or out of range")
            out[i] = c
    if (out == -1).any():
        raise RuntimeError("some frames were not processed by any rank")
    return out


def process_shard_packed(engine, frames, frame_ids, centers, lut, edge_cfg, mask_bits=None, edge_bits=None):
    """This rank's frames [n,H,W,3] (host, ideally pinned) through omni_host_color_edge_packed: the masks and edge planes of frame
    j land in mask_bits / edge_bits [j*K:(j+1)*K] (1 bit per pixel); returns ({frame_id: counts[K,3]}, result dict) for gather_counts.
    centers [K,3] / lut [K] are shared by all frames; centers [n,K,3] / lut [n,K] are this rank's frames' own (row j for frame j,
    e.g. the rows frame_ids select from per-frame centres of the whole batch)."""
    ids = [int(i) for i in frame_ids]
    if not ids:
        return {}, None
    c = np.asarray(centers)
    K = c.shape[1] if c.ndim == 3 else c.reshape(-1, 3).shape[0]
    if c.ndim == 3:
        centers, lut = c[:len(ids)], None if lut is None else np.asarray(lut)[:len(ids)]
    r = engine.host_color_edge_packed(frames[:len(ids)], centers, lut, edge_cfg, mask_bits=mask_bits, edge_bits=edge_bits)
    return {f: r["counts"][j * K:(j + 1) * K] for j, f in enumerate(ids)}, r
