"""Full-track separation by overlapping fixed-length segments, sharded across the ranks of one node.

The reference runs a whole track in one forward (inference/separate.py:135-148) and documents the OOMs that
follow (MEMORY_ANALYSIS.md:7-11); BASELINE config 3 instead cuts the track into 6-s segments at 50 % overlap,
each an independent forward, cross-faded with a periodic-Hann partition of unity (the first / last segment keep
a flat outer edge; the behaviour is defined once, in oracle/stitch.py).

Segments are the sharding unit.  Rank r owns a contiguous run of segments [lo, hi) and therefore the samples
[lo * half, hi * half) of the track (half = seg_len / 2; the last non-empty rank owns up to the end).  It
overlap-adds its segments (tfl_segment_ola) into a LOCAL buffer covering its own range plus a right halo of
`half` samples -- the second half of its last segment, which belongs to the next rank.  The exchange step is then
  1. halo:   rank r sends its right halo [S, half] (2.1 MB for 4 sources at 6-s segments) to the next non-empty
             rank, which adds it onto the first `half` samples of its own range (point-to-point, NCCL send/recv);
  2. gather: all-gather of the disjoint own ranges (padded to the longest) -- every rank ends with the full track.
No whole-track reduction, no pickled Python objects, no host synchronisation.

Any other overlap, or a [C, T] track, takes the general path: segments start every `hop` samples, the rows of all
channels of a batch of segments go through the model together ([b * C, L]), and tfl_segment_ola_hop stitches them
without atomics, normalised by the window sum of the covering segments.  Rank r owns [lo * hop, hi * hop) and its local
buffer runs to (hi - 1) * hop + L; the part past its own range can cover several later ranks, so each slice goes by
point-to-point to the rank that owns it before the same all-gather.
"""
import math
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch

from .engine import segment_ola, segment_ola_hop

SEGMENT_SAMPLES = 264600  # 6 s at 44.1 kHz


def segment_starts(n_samples: int, seg_len: int, hop: Optional[int] = None) -> List[int]:
    hop = hop or seg_len // 2
    n = max(1, math.ceil((n_samples - seg_len) / hop) + 1)
    return [i * hop for i in range(n)]


def partition(n_seg: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous block partition, larger blocks first: 79 over 8 -> 10,10,10,10,10,10,10,9."""
    base, extra = divmod(n_seg, world)
    out, lo = [], 0
    for r in range(world):
        hi = lo + base + (1 if r < extra else 0)
        out.append((lo, hi))
        lo = hi
    return out


def owned_ranges(n_seg: int, seg_len: int, world: int, hop: Optional[int] = None) -> List[Tuple[int, int]]:
    """Sample range [a, b) of the padded track each rank owns (empty for a rank without segments)."""
    hop = hop or seg_len // 2
    total = (n_seg - 1) * hop + seg_len
    parts = partition(n_seg, world)
    last = max(r for r, (lo, hi) in enumerate(parts) if hi > lo)
    out = []
    for r, (lo, hi) in enumerate(parts):
        if hi <= lo:
            out.append((0, 0))
        else:
            out.append((lo * hop, total if r == last else hi * hop))
    return out


def overlap_hop(seg_len: int, overlap: float) -> int:
    """Hop between segment starts for a fractional ``overlap`` in (0, 1): round(seg_len * (1 - overlap)), in [1, seg_len)."""
    if not 0.0 < overlap < 1.0:
        raise ValueError(f"overlap must be in (0, 1) (got {overlap})")
    if seg_len < 2:
        raise ValueError(f"segment length must be at least 2 samples (got {seg_len})")
    return min(seg_len - 1, max(1, round(seg_len * (1.0 - overlap))))


def separate_track(model: Callable[[torch.Tensor], Dict[str, torch.Tensor]], track: torch.Tensor,
                   seg_len: int = SEGMENT_SAMPLES, batch: int = 8, group=None, ola: Optional[Callable] = None,
                   names: Optional[Sequence[str]] = None, overlap: float = 0.5,
                   ola_hop: Optional[Callable] = None) -> Dict[str, torch.Tensor]:
    """track [T] mono or [C, T] (every rank holds it) -> {source: [T] or [C, T]} on every rank.

    ``model([rows, seg_len]) -> {name: [rows, seg_len]}``; ``batch`` segments go through it per call (``batch * C``
    rows for a [C, T] track).  Consecutive segments overlap by the fraction ``overlap`` of ``seg_len`` (hop:
    overlap_hop).  ``ola(seg_out[S, b, L], first_index, n_seg, acc[S, n], origin)`` accumulates windowed segments into
    a buffer that starts at sample ``origin`` of the track (default: the CUDA kernel behind tfl_segment_ola); it serves
    a 1-D track at 0.5 overlap and an even ``seg_len``.  Every other case stitches with
    ``ola_hop(seg_out[S, b * C, L], C, hop, first_index, n_seg, acc[S, C, n], origin)`` (default: the CUDA kernel behind
    tfl_segment_ola_hop).  ``names``: output keys, needed only by a rank that owns no segment (more ranks than
    segments); such a rank otherwise learns them from one forward of a silent segment.
    """
    if track.ndim not in (1, 2):
        raise ValueError(f"track must be [T] or [C, T] (got {tuple(track.shape)})")
    hop = overlap_hop(seg_len, overlap)
    if track.ndim == 1 and overlap == 0.5 and seg_len % 2 == 0:
        return _separate_half(model, track, seg_len, batch, group, ola, names)
    return _separate_hop(model, track, seg_len, hop, batch, group, ola_hop or segment_ola_hop, names)


def _separate_half(model, track, seg_len, batch, group, ola, names):
    import torch.distributed as dist
    ola = ola or segment_ola
    world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
    rank = dist.get_rank(group) if world > 1 else 0
    n_samples = track.shape[-1]
    half = seg_len // 2
    starts = segment_starts(n_samples, seg_len)
    n_seg = len(starts)
    total = starts[-1] + seg_len
    lo, hi = partition(n_seg, world)[rank]
    own = owned_ranges(n_seg, seg_len, world)
    a, b = own[rank]
    padded = torch.zeros(total, dtype=track.dtype, device=track.device)
    padded[:n_samples] = track
    non_empty = [r for r in range(world) if own[r][1] > own[r][0]]
    is_last = rank == non_empty[-1]
    local_len = (b - a) + (0 if (is_last or hi <= lo) else half)          # own range + right halo
    acc = None
    for i0 in range(lo, hi, batch):
        idx = range(i0, min(i0 + batch, hi))
        segs = torch.stack([padded[starts[i]:starts[i] + seg_len] for i in idx])
        out = model(segs)
        names = list(out.keys())
        seg_out = torch.stack([out[k] for k in names])            # [S, b, L]
        if acc is None:
            acc = torch.zeros(len(names), local_len, dtype=seg_out.dtype, device=seg_out.device)
        ola(seg_out, i0, n_seg, acc, a)
    if world == 1:
        return {k: acc[i, :n_samples] for i, k in enumerate(names)}
    if names is None:                                             # a rank without segments (world > n_seg)
        names = list(model(padded.new_zeros(1, seg_len)).keys())
    S = len(names)
    if acc is None:
        acc = torch.zeros(S, 0, dtype=torch.float32, device=track.device)
    # ---- 1. halo exchange between neighbouring non-empty ranks (point to point) ----
    if rank in non_empty:
        k = non_empty.index(rank)
        ops, recv = [], None
        if k + 1 < len(non_empty):
            send = acc[:, b - a:].contiguous()                    # [S, half]: belongs to the next rank
            ops.append(dist.P2POp(dist.isend, send, non_empty[k + 1], group))
        if k > 0:
            recv = torch.empty(S, half, dtype=acc.dtype, device=acc.device)
            ops.append(dist.P2POp(dist.irecv, recv, non_empty[k - 1], group))
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
        if recv is not None:
            acc[:, :half] += recv
    # ---- 2. all-gather of the disjoint own ranges (padded to the longest) ----
    longest = max(hi_ - lo_ for lo_, hi_ in own)
    mine = torch.zeros(S, longest, dtype=acc.dtype, device=acc.device)
    mine[:, : b - a] = acc[:, : b - a]
    parts = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(parts, mine, group=group)
    full = torch.empty(S, total, dtype=acc.dtype, device=acc.device)
    for r, (ra, rb) in enumerate(own):
        if rb > ra:
            full[:, ra:rb] = parts[r][:, : rb - ra]
    return {k: full[i, :n_samples] for i, k in enumerate(names)}


def _separate_hop(model, track, seg_len, hop, batch, group, ola_hop, names):
    import torch.distributed as dist
    world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
    rank = dist.get_rank(group) if world > 1 else 0
    x = track[None] if track.ndim == 1 else track                 # [C, T]
    C, n_samples = x.shape
    starts = segment_starts(n_samples, seg_len, hop)
    n_seg = len(starts)
    total = starts[-1] + seg_len
    parts = partition(n_seg, world)
    lo, hi = parts[rank]
    own = owned_ranges(n_seg, seg_len, world, hop)
    a, b = own[rank]
    ends = [(h - 1) * hop + seg_len if h > l else 0 for l, h in parts]  # end of each rank's local buffer
    padded = torch.zeros(C, total, dtype=x.dtype, device=x.device)
    padded[:, :n_samples] = x
    acc = None
    for i0 in range(lo, hi, batch):
        idx = range(i0, min(i0 + batch, hi))
        segs = torch.stack([padded[:, starts[i]:starts[i] + seg_len] for i in idx]).reshape(-1, seg_len)
        out = model(segs)                                         # rows: segment-major, channel-minor
        names = list(out.keys())
        seg_out = torch.stack([out[k] for k in names])            # [S, b * C, L]
        if acc is None:
            acc = torch.zeros(len(names), C, ends[rank] - a, dtype=seg_out.dtype, device=seg_out.device)
        ola_hop(seg_out, C, hop, i0, n_seg, acc, a)

    def result(full):
        return {k: (full[i, 0] if track.ndim == 1 else full[i])[..., :n_samples] for i, k in enumerate(names)}

    if world == 1:
        return result(acc)
    if names is None:                                             # a rank without segments (world > n_seg)
        names = list(model(padded.new_zeros(1, seg_len)).keys())
    S = len(names)
    if acc is None:
        acc = torch.zeros(S, C, 0, dtype=torch.float32, device=track.device)
    # ---- 1. the part of each local buffer past its own range, to every later rank that owns a slice of it ----
    ops, recvs = [], []
    if hi > lo:
        for r in range(rank + 1, world):
            ra, rb = own[r]
            if rb > ra and ra < ends[rank]:
                send = acc[:, :, ra - a:min(rb, ends[rank]) - a].contiguous()
                ops.append(dist.P2POp(dist.isend, send, r, group))
        for r in range(rank):
            if ends[r] > a:
                recv = torch.empty(S, C, min(b, ends[r]) - a, dtype=acc.dtype, device=acc.device)
                ops.append(dist.P2POp(dist.irecv, recv, r, group))
                recvs.append(recv)
    if ops:
        for req in dist.batch_isend_irecv(ops):
            req.wait()
    for recv in recvs:                                            # in rank order: the same sum on every run
        acc[:, :, :recv.shape[-1]] += recv
    # ---- 2. all-gather of the disjoint own ranges (padded to the longest) ----
    longest = max(hi_ - lo_ for lo_, hi_ in own)
    mine = torch.zeros(S, C, longest, dtype=acc.dtype, device=acc.device)
    mine[:, :, : b - a] = acc[:, :, : b - a]
    gathered = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(gathered, mine, group=group)
    full = torch.empty(S, C, total, dtype=acc.dtype, device=acc.device)
    for r, (ra, rb) in enumerate(own):
        if rb > ra:
            full[:, :, ra:rb] = gathered[r][:, :, : rb - ra]
    return result(full)
