"""Deterministic synthetic video streams (SURVEY.md §8(d)), integer arithmetic only.

Every value is produced by a counter-based 64-bit hash and integer interpolation, so the
frames are bit-identical on any machine / numpy build.  A stream is a smooth static
background plus one (or several) unblurred textured rectangles that move linearly and
reflect at the frame borders; the RGB composite is converted to NV12 with the BT.601
limited-range forward transform so that the reference's inverse transform
(/root/reference/src/nv12_convert.rs:24-30,124-126) applies.

This module is input generation only; it is not part of the tracker hot path.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Tuple

import numpy as np

_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def hash_u64(seed: int, n: int, offset: int = 0) -> np.ndarray:
    """splitmix64 of (seed, offset + i) for i in [0, n) -> uint64[n]."""
    with np.errstate(over="ignore"):
        idx = np.arange(offset, offset + n, dtype=np.uint64)
        z = idx * np.uint64(0x9E3779B97F4A7C15) + np.uint64(seed & 0xFFFFFFFFFFFFFFFF) * np.uint64(0xD1342543DE82EF95)
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return z


def hash_u8(seed: int, shape: Tuple[int, ...], offset: int = 0) -> np.ndarray:
    n = int(np.prod(shape))
    return (hash_u64(seed, n, offset) >> np.uint64(56)).astype(np.uint8).reshape(shape)


def rgb_to_nv12(rgb: np.ndarray) -> np.ndarray:
    """BT.601 limited-range RGB(HWC u8) -> NV12 bytes (tightly packed, len = w*h*3/2).

    Height and width must be even.  Chroma is taken from the rounded 2x2 mean of RGB.
    """
    h, w, _ = rgb.shape
    assert h % 2 == 0 and w % 2 == 0
    p = rgb.astype(np.int32)
    r, g, b = p[..., 0], p[..., 1], p[..., 2]
    y = ((66 * r + 129 * g + 25 * b + 128) >> 8) + 16
    m = (p[0::2, 0::2] + p[0::2, 1::2] + p[1::2, 0::2] + p[1::2, 1::2] + 2) >> 2
    mr, mg, mb = m[..., 0], m[..., 1], m[..., 2]
    u = ((-38 * mr - 74 * mg + 112 * mb + 128) >> 8) + 128
    v = ((112 * mr - 94 * mg - 18 * mb + 128) >> 8) + 128
    out = np.empty(w * h * 3 // 2, dtype=np.uint8)
    out[: w * h] = np.clip(y, 0, 255).astype(np.uint8).ravel()
    uv = np.empty((h // 2, w), dtype=np.uint8)
    uv[:, 0::2] = np.clip(u, 0, 255)
    uv[:, 1::2] = np.clip(v, 0, 255)
    out[w * h:] = uv.ravel()
    return out


def rgb_to_yuy2(rgb: np.ndarray) -> np.ndarray:
    """BT.601 limited-range RGB(HWC u8) -> packed YUY2 bytes (words Y0 U Y1 V, rows of 4 * ceil(w/2) bytes, len = 4 * ceil(w/2) * h).

    Any width and height.  Luma as rgb_to_nv12; chroma from the rounded mean of each horizontal pixel pair.  An odd width pads the
    last word with a copy of the last pixel (its chroma is that pixel's own, Y1 = Y0).
    """
    h, w, _ = rgb.shape
    p = rgb.astype(np.int32)
    if w % 2:
        p = np.concatenate([p, p[:, -1:]], axis=1)
    r, g, b = p[..., 0], p[..., 1], p[..., 2]
    y = np.clip(((66 * r + 129 * g + 25 * b + 128) >> 8) + 16, 0, 255)
    m = (p[:, 0::2] + p[:, 1::2] + 1) >> 1
    mr, mg, mb = m[..., 0], m[..., 1], m[..., 2]
    u = np.clip(((-38 * mr - 74 * mg + 112 * mb + 128) >> 8) + 128, 0, 255)
    v = np.clip(((112 * mr - 94 * mg - 18 * mb + 128) >> 8) + 128, 0, 255)
    out = np.empty((h, p.shape[1] // 2, 4), dtype=np.uint8)
    out[..., 0], out[..., 1], out[..., 2], out[..., 3] = y[:, 0::2], u, y[:, 1::2], v
    return out.reshape(-1)


def i420_layout(w: int, h: int) -> Tuple[int, int, int, int, int]:
    """GStreamer's default I420 layout: (Y stride, U / V stride, U offset, V offset, frame bytes)."""
    s0, s1, ch = (w + 3) & ~3, ((w + 1) // 2 + 3) & ~3, (h + 1) // 2
    u = s0 * (h + (h & 1))
    return s0, s1, u, u + s1 * ch, u + 2 * s1 * ch


def rgb_to_i420(rgb: np.ndarray) -> np.ndarray:
    """BT.601 limited-range RGB(HWC u8) -> planar I420 bytes in GStreamer's default layout (i420_layout): Y, then U, then V.

    Any width and height.  Luma and chroma as rgb_to_nv12 (the rounded 2x2 mean); at an odd size the last column / row is replicated
    into the missing half of its 2x2 blocks.  Row padding and the Y padding row of an odd height are zero.
    """
    h, w, _ = rgb.shape
    p = np.asarray(rgb, dtype=np.uint8)
    p = np.pad(p, ((0, h & 1), (0, w & 1), (0, 0)), mode="edge")
    nv = rgb_to_nv12(p)
    H2, W2 = p.shape[0], p.shape[1]
    s0, s1, uo, vo, n = i420_layout(w, h)
    out = np.zeros(n, dtype=np.uint8)
    out[: s0 * h].reshape(h, s0)[:, :w] = nv[: W2 * H2].reshape(H2, W2)[:h, :w]
    uv = nv[W2 * H2:].reshape(H2 // 2, W2 // 2, 2)
    out[uo: vo].reshape(H2 // 2, s1)[:, : W2 // 2] = uv[..., 0]
    out[vo:].reshape(H2 // 2, s1)[:, : W2 // 2] = uv[..., 1]
    return out


def _rgb_to_32(rgb: np.ndarray, pad, order) -> np.ndarray:
    h, w, _ = rgb.shape
    out = np.empty((h, w, 4), dtype=np.uint8)
    out[..., :3] = np.asarray(rgb, dtype=np.uint8)[..., order]
    out[..., 3] = np.broadcast_to(np.asarray(pad, dtype=np.uint8).reshape((h, w) if np.ndim(pad) else ()), (h, w))
    return out.reshape(-1)


def rgb_to_rgba(rgb: np.ndarray, pad=255) -> np.ndarray:
    """RGB(HWC u8) -> packed RGBA bytes R G B A (rows of 4 * w bytes, len = 4 * w * h).  `pad` is byte 3 of every pixel: a constant
    (255: an opaque alpha; any value: RGBx padding) or an array of h * w bytes."""
    return _rgb_to_32(rgb, pad, [0, 1, 2])


def rgb_to_bgra(rgb: np.ndarray, pad=255) -> np.ndarray:
    """RGB(HWC u8) -> packed BGRA bytes B G R A (rows of 4 * w bytes, len = 4 * w * h); `pad` as in rgb_to_rgba."""
    return _rgb_to_32(rgb, pad, [2, 1, 0])


def smooth_background(seed: int, w: int, h: int, cell: int = 32) -> np.ndarray:
    """Integer bilinear up-sampling of a coarse hash-noise grid plus 4-bit fine grain."""
    gh, gw = h // cell + 2, w // cell + 2
    grid = hash_u8(seed, (gh, gw, 3)).astype(np.int32)
    ys = np.arange(h)
    xs = np.arange(w)
    gy, fy = ys // cell, (ys % cell)[:, None, None]
    gx, fx = xs // cell, (xs % cell)[None, :, None]
    a = grid[gy][:, gx]
    b = grid[gy][:, gx + 1]
    c = grid[gy + 1][:, gx]
    d = grid[gy + 1][:, gx + 1]
    top = (cell - fx) * a + fx * b
    bot = (cell - fx) * c + fx * d
    val = ((cell - fy) * top + fy * bot + (cell * cell) // 2) // (cell * cell)
    grain = (hash_u8(seed ^ 0x5BD1E995, (h, w, 1)).astype(np.int32) & 15) - 8
    return np.clip(val + grain, 0, 255).astype(np.uint8)


@dataclass
class Target:
    x: int
    y: int
    w: int
    h: int
    vx: int
    vy: int
    texture: np.ndarray = field(repr=False, default=None)


@dataclass
class StreamSpec:
    name: str
    width: int
    height: int
    seed: int
    targets: List[Tuple[int, int, int, int, int, int]]  # (x, y, w, h, vx, vy)
    fmt: str = "nv12"  # "nv12" | "rgb24"


def _cfg4_targets() -> List[Tuple[int, int, int, int, int, int]]:
    out = []
    for i in range(16):
        gx, gy = i % 4, i // 4
        sx = 1 if (i % 2 == 0) else -1
        sy = 1 if ((i // 2) % 2 == 0) else -1
        out.append((380 + gx * 900, 220 + gy * 500, 200, 150, sx * (3 + i % 4), sy * (2 + i // 4)))
    return out


# The five configurations of BASELINE.json / SURVEY.md §8(d).
CONFIGS = {
    "cfg1": StreamSpec("cfg1", 1280, 720, 1001, [(580, 315, 120, 90, 5, 3)]),
    "cfg2": StreamSpec("cfg2", 1920, 1080, 1002, [(880, 480, 160, 120, 6, 3)]),
    "cfg3": StreamSpec("cfg3", 640, 512, 1003, [(288, 232, 64, 48, 3, 2)], fmt="rgb24"),
    "cfg4": StreamSpec("cfg4", 3840, 2160, 1004, _cfg4_targets()),
}


def cfg5_stream(i: int) -> StreamSpec:
    """Stream i (0..63) of cfg5: cfg2 geometry with seed 2000+i."""
    return StreamSpec(f"cfg5_{i}", 1920, 1080, 2000 + i, [(880, 480, 160, 120, 6, 3)])


class SyntheticStream:
    """Frame source: `frame(n)` returns frame n (NV12 bytes or HWC RGB24) deterministically."""

    def __init__(self, spec: StreamSpec):
        self.spec = spec
        w, h = spec.width, spec.height
        self.bg_rgb = smooth_background(spec.seed, w, h)
        self.targets: List[Target] = []
        for k, (x, y, tw, th, vx, vy) in enumerate(spec.targets):
            tex = hash_u8(spec.seed * 131 + 7 + k, (th, tw, 3))
            self.targets.append(Target(x, y, tw, th, vx, vy, tex))
        self._bg_nv12 = rgb_to_nv12(self.bg_rgb) if spec.fmt == "nv12" else None

    @staticmethod
    def _reflect(p0: int, v: int, n: int, lim: int) -> int:
        """Position after n steps of velocity v inside [0, lim] with mirror reflection."""
        if lim <= 0:
            return 0
        period = 2 * lim
        q = (p0 + v * n) % period
        return q if q <= lim else period - q

    def target_boxes(self, n: int) -> List[Tuple[int, int, int, int]]:
        s = self.spec
        out = []
        for t in self.targets:
            x = self._reflect(t.x, t.vx, n, s.width - t.w)
            y = self._reflect(t.y, t.vy, n, s.height - t.h)
            out.append((x, y, t.w, t.h))
        return out

    def frame_rgb(self, n: int) -> np.ndarray:
        img = self.bg_rgb.copy()
        for t, (x, y, tw, th) in zip(self.targets, self.target_boxes(n)):
            img[y:y + th, x:x + tw] = t.texture
        return img

    def frame(self, n: int) -> np.ndarray:
        s = self.spec
        if s.fmt == "rgb24":
            return self.frame_rgb(n)
        w, h = s.width, s.height
        out = self._bg_nv12.copy()
        yp = out[: w * h].reshape(h, w)
        uvp = out[w * h:].reshape(h // 2, w)
        for t, (x, y, tw, th) in zip(self.targets, self.target_boxes(n)):
            # re-encode the even-aligned bounding region of the pasted target
            x0, y0 = x & ~1, y & ~1
            x1, y1 = min(w, (x + tw + 1) & ~1), min(h, (y + th + 1) & ~1)
            reg = self.bg_rgb[y0:y1, x0:x1].copy()
            reg[y - y0:y - y0 + th, x - x0:x - x0 + tw] = t.texture
            enc = rgb_to_nv12(reg)
            rh, rw = y1 - y0, x1 - x0
            yp[y0:y1, x0:x1] = enc[: rw * rh].reshape(rh, rw)
            uvp[y0 // 2:y1 // 2, x0:x1] = enc[rw * rh:].reshape(rh // 2, rw)
        return out

    def frame_bytes(self) -> int:
        s = self.spec
        return s.width * s.height * 3 if s.fmt == "rgb24" else s.width * s.height * 3 // 2
