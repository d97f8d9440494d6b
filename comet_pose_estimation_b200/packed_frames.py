"""Frames of clips with different image sizes in one flat buffer, for ``TrackerPredictor.track_batch``.

The clips are ordered into **size groups** (one group per distinct (H, W), groups by increasing (H, W), sequences of a
group in batch order) and their real frames are copied, group by group, into one flat float32 buffer: frame f is
(3, H_f, W_f) contiguous at element ``frame_offset[f]``.  Nothing is padded to the largest size, so a batch that mixes
1080p clips with 512x512 clips holds each frame at its own size.  A group's frames are contiguous, so the encoder reads
a group as a zero-copy (F_g, 3, H, W) view; the patch encoder reads any frame through the offset and size tables
(``comet_shallow_encoder_from_images_packed_f32``).

Clips that share frames of a video (``track_batch(clip_frames=...)``) are served from one such buffer too:
:func:`pack_referenced_frames` packs each distinct referenced frame once, and the clips read it through a frame table."""
from __future__ import annotations

import bisect
from typing import List, Sequence, Tuple

import torch


class PackedFrames:
    """``data`` (total,) float32; ``frame_offset`` (F,) int64 element offsets and ``frame_hw`` (F, 2) int32 (H, W) on the
    CPU (``device_tables()`` gives them on the data's device); per sequence b (batch order) ``seq_first[b]`` its first
    packed frame, ``seq_frames[b]`` its frame count and ``seq_hw[b]`` its (H, W); ``groups`` a list of
    ``((H, W), sequences)`` in packed order, ``group_first`` / ``group_frames`` the frame range of each group."""

    def __init__(self, clips: Sequence[torch.Tensor]):
        """``clips``: B tensors (S_b, 3, H_b, W_b), any strides (views of a padded tensor included); only their
        elements are read, each once."""
        assert len(clips) >= 1, "no clips"
        B = len(clips)
        self.seq_hw: List[Tuple[int, int]] = [(int(c.shape[2]), int(c.shape[3])) for c in clips]
        self.seq_frames: List[int] = [int(c.shape[0]) for c in clips]
        order = sorted(set(self.seq_hw))
        self.groups = [(hw, [b for b in range(B) if self.seq_hw[b] == hw]) for hw in order]
        self.seq_first = [0] * B
        self.group_first, self.group_frames = [], []
        offsets, hws, at = [], [], 0
        for hw, seqs in self.groups:
            self.group_first.append(len(hws))
            for b in seqs:
                self.seq_first[b] = len(hws)
                for _ in range(self.seq_frames[b]):
                    offsets.append(at)
                    hws.append(hw)
                    at += 3 * hw[0] * hw[1]
            self.group_frames.append(len(hws) - self.group_first[-1])
        self.frame_offset = torch.tensor(offsets, dtype=torch.int64)
        self.frame_hw = torch.tensor(hws, dtype=torch.int32).reshape(-1, 2)
        self.data = torch.empty(at, dtype=torch.float32, device=clips[0].device)
        for _, seqs in self.groups:
            for b in seqs:
                self.clip(b).copy_(clips[b])
        self._dev = None

    @property
    def num_frames(self) -> int:
        return int(self.frame_offset.shape[0])

    @property
    def device(self):
        return self.data.device

    def frames(self, first: int, count: int) -> torch.Tensor:
        """Packed frames [first, first + count), all of one size: a (count, 3, H, W) view of the buffer."""
        H, W = (int(v) for v in self.frame_hw[first])
        off = int(self.frame_offset[first])
        return self.data[off:off + count * 3 * H * W].view(count, 3, H, W)

    def clip(self, b: int) -> torch.Tensor:
        """Sequence b's frames: a (S_b, 3, H_b, W_b) view."""
        return self.frames(self.seq_first[b], self.seq_frames[b])

    def group(self, g: int) -> torch.Tensor:
        """The frames of size group g, sequence after sequence: a (F_g, 3, H_g, W_g) view."""
        return self.frames(self.group_first[g], self.group_frames[g])

    def device_tables(self):
        """(frame_offset int64 (F,), frame_hw int32 (F, 2)) on the data's device, uploaded once."""
        if self._dev is None:
            self._dev = (self.frame_offset.to(self.device), self.frame_hw.to(self.device).contiguous())
        return self._dev


def pack_referenced_frames(videos: Sequence[torch.Tensor], clip_frames: Sequence[Sequence[int]]):
    """The distinct frames that clips reference, packed once.  ``videos``: V tensors (T_v, 3, H_v, W_v) whose frames are
    numbered one after another, video 0 first; ``clip_frames``: B lists of frame numbers (validated).  The referenced
    frames are cut into runs of consecutive frames of one video; each run is a zero-copy view of its video and is copied
    into the buffer once, so frames that no clip references are never read.  -> (``PackedFrames`` whose "sequences" are
    the runs, ``ids``: B lists, ``ids[b][s]`` the packed frame of ``clip_frames[b][s]``)."""
    first = [0]
    for v in videos:
        first.append(first[-1] + int(v.shape[0]))
    runs = []                                          # [video, first frame in the video, count]
    for t in sorted({t for c in clip_frames for t in c}):
        v = bisect.bisect_right(first, t) - 1
        if runs and runs[-1][0] == v and runs[-1][1] + runs[-1][2] == t - first[v]:
            runs[-1][2] += 1
        else:
            runs.append([v, t - first[v], 1])
    packed = PackedFrames([videos[v][t0:t0 + n] for v, t0, n in runs])
    packed_of = {first[v] + t0 + k: packed.seq_first[r] + k for r, (v, t0, n) in enumerate(runs) for k in range(n)}
    return packed, [[packed_of[t] for t in c] for c in clip_frames]
