"""numpy model of the calm analysis of the unsharp stage (DESIGN.md §5.1; kernels_pyramid.cu EmitCtx,
kernels_unsharp.cu k_calm_scan / k_calm_blocks / k_calm_chunks / launch_calm_analysis).

From a frame's float lapBlend x (H x W x 3, as STAGE_LAP_BLEND returns it) the model computes what the calm route
decides: the emitted bytes q, the clamp-excess flags, the per-block second-difference maxima hx / hy, the block flags,
the strip-chunk flags that select the exact unsharp pass and the level-0 collapse tiles that pass reads. The tests
compare it with the kernels (flag counts) and with the CPU restatement of unsharp_mask (soundness of the bound). The
constants are read from the sources, so a change there changes the model too."""
from __future__ import annotations

import os
import re
from dataclasses import dataclass

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEVICE = os.path.join(ROOT, "poppy_b200", "csrc", "device")


def _source(*parts) -> str:
    with open(os.path.join(ROOT, *parts)) as f:
        return f.read()


def _int_const(text: str, name: str) -> int:
    m = re.search(r"\b" + name + r"\s*=\s*(\d+)\s*[;,]", text)
    assert m, name
    return int(m.group(1))


_UNSHARP = _source("poppy_b200", "csrc", "device", "kernels_unsharp.cu")
_KERNELS_H = _source("poppy_b200", "csrc", "device", "kernels.cuh")
CALM_SUM = _int_const(_UNSHARP, "CALM_SUM")
STRIP_W = _int_const(_UNSHARP, "US_W")
BLOCK_W = _int_const(_KERNELS_H, "CALM_BLOCK_W")
BLOCK_H = _int_const(_KERNELS_H, "CALM_BLOCK_H")
CHUNK_ROWS = _int_const(_source("poppy_b200", "csrc", "poppy_cuda.cu"), "kSparseChunkRows")
EMIT_EXCESS_TOL = np.float32(float(re.search(r"EMIT_EXCESS_TOL\s*=\s*([0-9.]+)f",
                                             _source("poppy_b200", "csrc", "device", "kernels_pyramid.cu")).group(1)))
TILE_W, TILE_H = 128, 32            # level-0 collapse tiles (k_collapse_tma / k_collapse_roll CTAs)
NORM_T = 0.3                        # unsharp_mask threshold (src/util.cpp:135)


def div_up(a: int, b: int) -> int:
    return -(-a // b)


def force_all(w: int, h: int) -> bool:
    """launch_calm_analysis skips the byte scan and flags every chunk (the frame ring itself is word aligned)."""
    return w % 4 != 0 or w < 8 or h < 2


def emit(x: np.ndarray):
    """The fused level-0 store: q = sat(cvRound(255 x)) and per channel the clamp excess |255 x - clamp(255 x)|."""
    t = x.astype(np.float32) * np.float32(255.0)
    cl = np.clip(t, np.float32(0.0), np.float32(255.0))
    return np.rint(cl).astype(np.uint8), np.abs(t - cl)


def _block_max(a: np.ndarray) -> np.ndarray:
    """Max over 4 x 8 blocks (and the channel axis, if any) of an H x W (x C) array; partial blocks at the edges."""
    h, w = a.shape[:2]
    bh, bw = div_up(h, BLOCK_H), div_up(w, BLOCK_W)
    pad = np.zeros((bh * BLOCK_H, bw * BLOCK_W) + a.shape[2:], a.dtype)
    pad[:h, :w] = a
    pad = pad.reshape(bh, BLOCK_H, bw, BLOCK_W, -1)
    return pad.max(axis=(1, 3, 4))


def second_dev(q: np.ndarray):
    """Per pixel and channel |floor((q[-1] + q[+1]) / 2) - q| along x and along y, neighbours reflected at the image
    border (BORDER_REFLECT_101, numpy's 'reflect')."""
    qi = q.astype(np.int32)
    px = np.pad(qi, ((0, 0), (1, 1), (0, 0)), mode="reflect")
    py = np.pad(qi, ((1, 1), (0, 0), (0, 0)), mode="reflect")
    dx = np.abs((px[:, :-2] + px[:, 2:]) // 2 - qi)
    dy = np.abs((py[:-2] + py[2:]) // 2 - qi)
    return dx, dy


def _nbhd_max(t: np.ndarray, rx: int, ry: int) -> np.ndarray:
    """Max over the blocks within rx block columns / ry block rows (clipped to the table)."""
    bh, bw = t.shape
    pad = np.full((bh + 2 * ry, bw + 2 * rx), -1, np.int32)
    pad[ry:ry + bh, rx:rx + bw] = t
    out = np.full((bh, bw), -1, np.int32)
    for dy in range(2 * ry + 1):
        for dx in range(2 * rx + 1):
            np.maximum(out, pad[dy:dy + bh, dx:dx + bw], out=out)
    return out


@dataclass
class CalmAnalysis:
    q: np.ndarray              # H x W x 3 emitted bytes
    excess: np.ndarray         # bh x bw x 3: the block's clamp excess exceeds EMIT_EXCESS_TOL
    hx: np.ndarray             # bh x bw (255 where a channel's excess flag is set)
    hy: np.ndarray
    nbhd: np.ndarray           # bh x bw: max hx + max hy over the block neighbourhood
    block_flags: np.ndarray    # bh x bw bool
    chunk_flags: np.ndarray    # chunks_y x strips bool
    tile_flags: np.ndarray     # ceil(h/32) x ceil(w/128) bool
    forced: bool

    @property
    def flagged_chunks(self) -> int:
        return int(self.chunk_flags.sum())

    def pixel_block_flags(self) -> np.ndarray:
        """H x W: the block of the pixel is flagged."""
        h, w = self.q.shape[:2]
        return np.repeat(np.repeat(self.block_flags, BLOCK_H, 0), BLOCK_W, 1)[:h, :w]

    def pixel_chunk_flags(self) -> np.ndarray:
        h, w = self.q.shape[:2]
        return np.repeat(np.repeat(self.chunk_flags, CHUNK_ROWS, 0), STRIP_W, 1)[:h, :w]

    def pixel_nbhd(self) -> np.ndarray:
        h, w = self.q.shape[:2]
        return np.repeat(np.repeat(self.nbhd, BLOCK_H, 0), BLOCK_W, 1)[:h, :w]


def chunk_and_tile_flags(block_flags: np.ndarray, w: int, h: int, forced: bool, chunk_rows: int = CHUNK_ROWS,
                         col_margin=(8, 128), row_margin=(5, 5)):
    """k_calm_chunks: a strip chunk (120 columns x chunk_rows rows) is flagged when one of its blocks is; a flagged chunk
    flags the level-0 collapse tiles holding columns x0-8 .. x0+127 and rows Y0-5 .. Y1+4 (clipped), which
    k_unsharp_strip stages for it."""
    strips, chunks_y = div_up(w, STRIP_W), div_up(h, chunk_rows)
    chunks = np.zeros((chunks_y, strips), bool)
    tiles = np.zeros((div_up(h, TILE_H), div_up(w, TILE_W)), bool)
    for cy in range(chunks_y):
        y0, y1 = cy * chunk_rows, min(cy * chunk_rows + chunk_rows, h)
        for sx in range(strips):
            x0, x1 = sx * STRIP_W, min(sx * STRIP_W + STRIP_W, w)
            any_ = forced or bool(block_flags[y0 // BLOCK_H:(y1 - 1) // BLOCK_H + 1, x0 // BLOCK_W:(x1 - 1) // BLOCK_W + 1].any())
            chunks[cy, sx] = any_
            if any_:
                tx0, tx1 = max(x0 - col_margin[0], 0) // TILE_W, (min(x0 + col_margin[1], w) - 1) // TILE_W
                ty0, ty1 = max(y0 - row_margin[0], 0) // TILE_H, (min(y1 + row_margin[1], h) - 1) // TILE_H
                tiles[ty0:ty1 + 1, tx0:tx1 + 1] = True
    return chunks, tiles


def analyse(x: np.ndarray, calm_sum: int = CALM_SUM, rx: int = 2, ry: int = 1, tol=EMIT_EXCESS_TOL) -> CalmAnalysis:
    """The calm analysis of one frame's lapBlend x (H x W x 3 float32)."""
    h, w = x.shape[:2]
    q, ex = emit(x)
    forced = force_all(w, h)
    excess = np.stack([_block_max(ex[..., c]) for c in range(3)], -1) > tol
    dx, dy = second_dev(q)
    hx, hy = _block_max(dx).astype(np.int32), _block_max(dy).astype(np.int32)
    ex_any = excess.any(-1)
    hx[ex_any] = 255
    hy[ex_any] = 255
    nbhd = _nbhd_max(hx, rx, ry) + _nbhd_max(hy, rx, ry)
    block_flags = nbhd > calm_sum
    if forced:
        block_flags = np.ones_like(block_flags)
    chunks, tiles = chunk_and_tile_flags(block_flags, w, h, forced)
    return CalmAnalysis(q, excess, hx, hy, nbhd, block_flags, chunks, tiles, forced)


def fired(x: np.ndarray, sharp: np.ndarray) -> np.ndarray:
    """H x W: unsharp_mask changed the pixel (the 3x3 median reached the threshold and moved some channel)."""
    return (x.view(np.uint32) != sharp.view(np.uint32)).any(-1)
