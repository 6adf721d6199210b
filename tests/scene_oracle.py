"""numpy fp32 restatement of the whole-scan contract of include/r3dfs.h ("Segmenting a whole scan"):
grid, block memberships, chunk layout, chunk clouds and the merge of chunk logits.  Every float
operation is a single numpy float32 operation, rounded to nearest as the CUDA code's __fsub_rn /
__fdiv_rn / __fadd_rn, so the GPU results are compared with torch.equal, not a tolerance."""
from __future__ import annotations

import numpy as np

F32 = np.float32


def lowbias32(x):
    x = np.asarray(x, dtype=np.uint64) & 0xFFFFFFFF
    x ^= x >> 16
    x = (x * 0x7FEB352D) & 0xFFFFFFFF
    x ^= x >> 15
    x = (x * 0x846CA68B) & 0xFFFFFFFF
    x ^= x >> 16
    return x


def _axis(c, stride, r):
    """cell of every point, and the block range [lo, hi] of every point along one axis"""
    c0 = c.min()
    ext = F32(c.max() - c0)
    q = np.floor(F32(F32(ext / stride) + F32(0.5)))
    n_cells = max(1, int(q))
    u = np.minimum(np.floor((c - c0) / stride).astype(np.int64), n_cells - 1)
    n_blocks = max(1, n_cells - r + 1)
    return u, np.maximum(0, u - r + 1), np.minimum(u, n_blocks - 1), n_cells, n_blocks


def plan(points, n_points, block_size=1.0, overlap=1, seed=0):
    """-> dict(chunk_src (E, N) int32, chunk_x (E, N, 9) float32, mem_point / mem_chunk / mem_slot
    (memberships in point order, within a point ascending block id), coverage (M,), grid sizes)."""
    pts = np.asarray(points, dtype=F32)
    M, N, r = pts.shape[0], int(n_points), int(overlap)
    stride = F32(F32(block_size) / F32(r))
    ux, lox, hix, ncx, nbx = _axis(pts[:, 0], stride, r)
    uy, loy, hiy, ncy, nby = _axis(pts[:, 1], stride, r)
    P, B = [], []
    for dx in range(r):
        for dy in range(r):
            ix, iy = lox + dx, loy + dy
            ok = (ix <= hix) & (iy <= hiy)
            P.append(np.nonzero(ok)[0])
            B.append((ix * nby + iy)[ok])
    P, B = np.concatenate(P), np.concatenate(B)
    o = np.lexsort((B, P))                      # point order, then ascending block id
    P, B = P[o], B[o]
    key = lowbias32(P.astype(np.uint64) ^ lowbias32(int(seed) & 0xFFFFFFFF))
    srt = np.lexsort((key, B))                  # by (block, key)
    Bs = B[srt]
    blocks, start, n_b = np.unique(Bs, return_index=True, return_counts=True)
    cb = (n_b + N - 1) // N
    chunk_off = np.concatenate([[0], np.cumsum(cb)])
    seg = np.repeat(np.arange(len(blocks)), n_b)
    rho = np.arange(len(Bs)) - start[seg]
    mem_chunk = np.empty(len(P), np.int64)
    mem_slot = np.empty(len(P), np.int64)
    mem_chunk[srt] = chunk_off[seg] + rho % cb[seg]
    mem_slot[srt] = rho // cb[seg]
    E = int(chunk_off[-1])
    cseg = np.repeat(np.arange(len(blocks)), cb)
    j = np.arange(E) - chunk_off[cseg]
    count = (n_b[cseg] - j + cb[cseg] - 1) // cb[cseg]
    q = np.arange(N)[None, :]
    sp = q % count[:, None]
    src = P[srt][start[cseg][:, None] + sp * cb[cseg][:, None] + j[:, None]]
    xyz = pts[src, 0:3]
    m = xyz.min(1, keepdims=True)
    xyzp = xyz - m
    e = xyzp.max(1, keepdims=True)
    XYZ = np.where(e > 0, xyzp / np.where(e > 0, e, F32(1)), F32(0)).astype(F32)
    rgb = pts[src, 3:6] / F32(255)
    chunk_x = np.concatenate([xyzp, rgb, XYZ], 2).astype(F32)
    coverage = np.bincount(P, minlength=M)
    return dict(chunk_src=src.astype(np.int32), chunk_x=chunk_x, mem_point=P, mem_block=B,
                mem_chunk=mem_chunk, mem_slot=mem_slot, coverage=coverage, n_chunks=E,
                cells=(ncx, ncy), blocks=(nbx, nby), cell=(ux, uy), count=count)


def merge(logits, pl):
    """Chunk logits (E, N, nc) -> (point logits (M, nc) float32, pred (M,), coverage (M,))."""
    logits = np.asarray(logits, dtype=F32)
    P, c, s = pl["mem_point"], pl["mem_chunk"], pl["mem_slot"]
    M, nc = len(pl["coverage"]), logits.shape[2]
    acc = np.zeros((M, nc), F32)
    first = np.concatenate([[0], np.cumsum(pl["coverage"])[:-1]])
    ordinal = np.arange(len(P)) - first[P]      # k-th membership of its point
    for k in range(int(ordinal.max()) + 1):
        sel = ordinal == k
        acc[P[sel]] = acc[P[sel]] + logits[c[sel], s[sel]]
    cov = pl["coverage"]
    out = (acc / cov.astype(F32)[:, None]).astype(F32)
    return out, out.argmax(1).astype(np.int32), cov.astype(np.int32)
