"""plot(c, imgpointss, n_corners, checker_size, sz): src/plot_calibration.jl:24-44.

The reference's debug output: every calibration image rectified with its own extrinsic, red
crosses on the detected corners (drawn before the warp), blue crosses on their rectified
world positions (drawn after it), saved under `debug/`.  The loop over files becomes ONE
cc_rectify_u8c3_views call; JPEG inputs are decoded on the device (cc_jpeg_decode_u8c3), other
formats (the reference's PNG examples) are read by OpenCV on the host like FileIO does.
"""
from __future__ import annotations

import os

import numpy as np

from .calibration import Calibration, image_transformations, warp_views, load_jpegs

try:
    import torch
except Exception:  # pragma: no cover
    torch = None

RED, BLUE = (255, 0, 0), (0, 0, 255)


def _draw_crosses(frame, points_rc, n1, color, origin=(1, 1)):
    """draw_crosses!, src/plot_calibration.jl:24-28.  frame: (sz2, sz1, 3) uint8 in the frame layout
    (frame[c, r] = pixel (r, c)); points_rc: (n, 2) 1-based (row, col) in the axes whose first index is
    origin; radius relative to the board's apparent size."""
    ij = np.rint(np.asarray(points_rc, dtype=np.float64)).astype(np.int64)
    radius = int(np.rint(np.linalg.norm((ij[0] - ij[n1 - 1]).astype(np.float64)) / n1 / 5))
    sz2, sz1 = frame.shape[:2]
    for r, c in ij:
        r0, c0 = r - origin[0], c - origin[1]                  # 0-based array position
        if 0 <= c0 < sz2:
            lo, hi = max(0, r0 - radius), min(sz1 - 1, r0 + radius)
            if lo <= hi:
                frame[c0, lo:hi + 1] = color
        if 0 <= r0 < sz1:
            lo, hi = max(0, c0 - radius), min(sz2 - 1, c0 + radius)
            if lo <= hi:
                frame[lo:hi + 1, r0] = color


def _load_rgb_frames(files, sz):
    """RGB.(FileIO.load(file)) for every file -> uint8 (n, sz2, sz1, 3) in the frame layout, on the host."""
    import cv2
    out = np.empty((len(files), sz[1], sz[0], 3), dtype=np.uint8)
    for i, f in enumerate(files):
        img = cv2.imread(f, cv2.IMREAD_COLOR)
        if img is None or img.shape[:2] != (sz[0], sz[1]):
            raise ValueError(f"{f}: cannot read an image of size {sz}")
        out[i] = img[:, :, ::-1].transpose(1, 0, 2)            # BGR (rows, cols) -> RGB [c][r]
    return out


def plot(c: Calibration, imgpointss, n_corners, checker_size, sz, dir="debug", coord="f64"):
    """Returns the list of files written.  imgpointss: (nfiles, n1*n2, 2), corner a fastest (detect_fit)."""
    import cv2
    os.makedirs(dir, exist_ok=True)
    n1 = int(n_corners[0])
    files = list(c.files)
    ips = np.asarray(imgpointss, dtype=np.float64)
    jpeg = all(f.lower().endswith((".jpg", ".jpeg")) for f in files)
    if jpeg:                                                   # decoded on the device (nvJPEG), no host decoder involved
        frames = load_jpegs(files).cpu().numpy()
    else:
        frames = _load_rgb_frames(files, sz)
    for i in range(len(files)):
        _draw_crosses(frames[i], ips[i], n1, RED)
    tf = [image_transformations(c, i, ips, checker_size, n_corners, sz) for i in range(len(files))]
    # host frames: one pipelined call over all views (cc_rectify_views_u8c3_host)
    warped = warp_views(c, list(range(len(files))), frames, [t[0] for t in tf], [t[1] for t in tf],
                        fill=(0, 0, 0), coord=coord)
    written = []
    for i, f in enumerate(files):
        ratio, axs = tf[i]
        world = c(ips[i], i)                                   # itform = s . pop . image2real
        _draw_crosses(warped[i], np.asarray(world)[:, :2] * ratio, n1, BLUE, origin=axs)
        path = os.path.join(dir, os.path.splitext(os.path.basename(f))[0] + ".png")
        cv2.imwrite(path, np.ascontiguousarray(warped[i].transpose(1, 0, 2)[:, :, ::-1]))
        written.append(path)
    return written
