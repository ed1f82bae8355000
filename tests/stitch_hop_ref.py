"""Full-track stitch at any overlap, and over channels -- TEST INFRASTRUCTURE ONLY.

``oracle/stitch.py`` defines the 50 %-overlap stitch; this module generalises it to any hop
0 < hop < seg_len and states what segments.separate_track computes off the default path:

  starts   s_i = i * hop, i = 0 .. n-1, n = max(1, ceil((T - seg_len) / hop) + 1)
  window   w_i: oracle.segment_window (periodic Hann; the first segment flat for m < seg_len // 2,
           the last for m >= seg_len // 2)
  output   y[t] = sum_i w_i[t - s_i] f_i[t - s_i] / E[t],  E[t] = sum_i w_i[t - s_i] over the segments
           covering t (E > 0 for every hop < seg_len; E == 1 at hop = seg_len / 2, where this is
           oracle.stitch_segments)
  channels a [C, T] track is segmented and stitched channel by channel.
"""
import math
from typing import Callable, Dict, List

import torch

from oracle import segment_window


def segment_starts(n_samples: int, seg_len: int, hop: int) -> List[int]:
    n = max(1, math.ceil((n_samples - seg_len) / hop) + 1)
    return [i * hop for i in range(n)]


def stitch_segments(seg_out: torch.Tensor, n_samples: int, hop: int) -> torch.Tensor:
    """seg_out [n_seg, n_src, seg_len] at starts i * hop -> [n_src, n_samples]."""
    n_seg, n_src, seg_len = seg_out.shape
    assert 0 < hop < seg_len
    starts = segment_starts(n_samples, seg_len, hop)
    assert len(starts) == n_seg
    total = starts[-1] + seg_len
    y = torch.zeros(n_src, total, dtype=seg_out.dtype)
    e = torch.zeros(total, dtype=seg_out.dtype)
    for i, s in enumerate(starts):
        w = segment_window(seg_len, i == 0, i == n_seg - 1, seg_out.dtype)
        y[:, s:s + seg_len] += seg_out[i] * w
        e[s:s + seg_len] += w
    return (y / e)[:, :n_samples]


def separate_track(forward: Callable[[torch.Tensor], Dict[str, torch.Tensor]], track: torch.Tensor,
                   seg_len: int, hop: int, batch: int = 1) -> Dict[str, torch.Tensor]:
    """track [T] or [C, T] -> {name: [T] or [C, T]} using ``forward([b, seg_len]) -> {name: [b, seg_len]}``."""
    if track.ndim == 1:
        return {k: v[0] for k, v in separate_track(forward, track[None], seg_len, hop, batch).items()}
    n_samples = track.shape[-1]
    starts = segment_starts(n_samples, seg_len, hop)
    padded = torch.zeros(track.shape[0], starts[-1] + seg_len, dtype=track.dtype)
    padded[:, :n_samples] = track
    per_channel = []
    for ch in padded:
        segs = torch.stack([ch[s:s + seg_len] for s in starts])
        outs, names = [], None
        for i in range(0, len(starts), batch):
            res = forward(segs[i:i + batch])
            names = list(res.keys())
            outs.append(torch.stack([res[k] for k in names], dim=1))
        y = stitch_segments(torch.cat(outs, dim=0), n_samples, hop)
        per_channel.append({k: y[i] for i, k in enumerate(names)})
    return {k: torch.stack([p[k] for p in per_channel]) for k in per_channel[0]}
