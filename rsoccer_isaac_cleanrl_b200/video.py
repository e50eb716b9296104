"""Frames to pictures and videos: a device-side mosaic of several fields and an mp4 writer.

The frames themselves come from the engine (`Engine.render`, include/vss_b200.h: vss_render). OpenCV is only
imported when a video is written, so the rest of the package does not need it.
"""
import math
import os
import re

import numpy as np
import torch

FPS = 20  # round(1 / dt) at the engine's control step dt = 0.05 s
HEIGHT, WIDTH = 560, 720  # the frame size of the videos (Engine.render's default): 400 px/m


def mosaic(frames):
    """(F, H, W, 3) frames laid out as a grid of ceil(sqrt(F)) columns, row by row, on the frames' device;
    tiles past the last frame are black. Returns (rows * H, cols * W, 3)."""
    f, h, w, c = frames.shape
    cols = math.ceil(math.sqrt(f))
    rows = math.ceil(f / cols)
    grid = frames.new_zeros((rows * cols, h, w, c))
    grid[:f] = frames
    return grid.view(rows, cols, h, w, c).permute(0, 2, 1, 3, 4).reshape(rows * h, cols * w, c)


def safe_name(name):
    """A team name as a file-name component: anything but letters, digits, '.', '-' and '_' becomes '_'."""
    return re.sub(r"[^A-Za-z0-9._-]", "_", str(name)).strip(".") or "_"


class VideoWriter:
    """Writes RGB frames (H, W, 3) uint8 to an mp4 (OpenCV, codec mp4v) at `fps` frames per second. Frames may be
    numpy arrays or tensors (copied to the host); the size is fixed by the first frame."""

    def __init__(self, path, fps=FPS):
        self.path, self.fps = path, fps
        self._w = None
        self.frames = 0

    def write(self, frame):
        if isinstance(frame, torch.Tensor):
            frame = frame.cpu().numpy()
        frame = np.ascontiguousarray(frame)
        if frame.dtype != np.uint8 or frame.ndim != 3 or frame.shape[2] != 3:
            raise ValueError(f"expected an (H, W, 3) uint8 frame, got {frame.dtype} {frame.shape}")
        import cv2
        if self._w is None:
            d = os.path.dirname(os.path.abspath(self.path))
            os.makedirs(d, exist_ok=True)
            self._w = cv2.VideoWriter(self.path, cv2.VideoWriter_fourcc(*"mp4v"), float(self.fps),
                                      (frame.shape[1], frame.shape[0]))
            if not self._w.isOpened():
                raise RuntimeError(f"OpenCV cannot open {self.path} for writing (mp4v)")
            self._size = frame.shape
        elif frame.shape != self._size:
            raise ValueError(f"frame size {frame.shape} differs from the video's {self._size}")
        self._w.write(cv2.cvtColor(frame, cv2.COLOR_RGB2BGR))
        self.frames += 1

    def write_frames(self, frames):
        """Writes (K, F, H, W, 3) or (K, H, W, 3) frames: one video frame per step k (several fields as a mosaic).
        One device-to-host copy for all K."""
        if not isinstance(frames, torch.Tensor):
            frames = torch.from_numpy(np.ascontiguousarray(frames))
        if frames.ndim == 5:
            frames = frames[:, 0] if frames.shape[1] == 1 else torch.stack([mosaic(fr) for fr in frames])
        for fr in frames.cpu().numpy():
            self.write(fr)

    def close(self):
        if self._w is not None:
            self._w.release()
            self._w = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
