"""Which items and respondents the benchmark-shape tests compare with the oracle, and the oracle references they share.

A kernel fault is usually confined to one tile: a ragged last tile, one column group of a tile schedule, one piece of a
chunked copy.  A few dozen random indices miss most such tiles at C3 and C5 ((1 - tile / size)^samples: a 64-item
tile of the fixed-point products escapes 32 random items 81 % of the time at C3, 90 % at C5).  The strata below put an
index in every tile instead, so a fault in any one tile reaches a compared value.  The tile sizes are restated below,
each with the kernel it comes from."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np

DG_BN = 64                  # item columns per output tile of k_dgemm_i8 (gpirt_b200/csrc/dgemm_i8.cu): nu = L Z, f* = A^T f
TI_BM = 128                 # respondents per row tile of k_igemm_theta (gpirt_b200/csrc/theta_int8.cu)
UPLOAD_PIECE = 32 << 20     # bytes per piece of the chunked upload of y (PIECE in upload_pageable, gpirt_b200/csrc/sampler.cu)
CHOL_NB = 128               # rows per panel of the factorisation (gpirt_b200/csrc/linalg.cuh)


def tile_strata(size, tile, both_ends):
    """both_ends: the first and the last index of every tile (the last tile may be ragged); otherwise one index per
    tile, alternating first and last, plus size - 1"""
    first = np.arange(0, size, tile)
    last = np.minimum(first + tile, size) - 1
    if both_ends:
        return np.unique(np.r_[first, last])
    return np.unique(np.r_[np.where(np.arange(first.size) % 2 == 0, first, last), size - 1])


def items(m, big):
    """C3 (big False): first and last item of every 64-item tile; C5: one per tile, alternating, plus m - 1"""
    return tile_strata(m, DG_BN, not big)


def respondents(n, big):
    """C3: first and last respondent of every 128-row tile; C5: one per tile, alternating, plus n - 1"""
    return tile_strata(n, TI_BM, not big)


def panel_rows(n):
    """first and last row of every 128-row panel of the factorisation"""
    return tile_strata(n, CHOL_NB, True)


def upload_pieces(n, m, cols):
    """(pieces of the chunked upload of the n x m float64 y that hold part of a column in `cols`, number of pieces).
    Pieces are of bytes: where y has missing cells they are NaN doubles, so the pieces do not depend on the share missing."""
    cols = np.asarray(cols, dtype=np.int64)
    col_bytes = 8 * int(n)
    total = -(-col_bytes * int(m) // UPLOAD_PIECE)
    first = cols * col_bytes // UPLOAD_PIECE
    last = ((cols + 1) * col_bytes - 1) // UPLOAD_PIECE
    hit = set()
    for a, b in zip(first, last):
        hit.update(range(int(a), int(b) + 1))
    return hit, total


def keyed_normals(O, seed, sweep, purpose, cols, n):
    """n x len(cols) oracle normals: column c holds the variates of stream cols[c], indices 0..n-1 (gpo_rng.h)"""
    z = np.empty((n, len(cols)), order="F")
    for c, j in enumerate(cols):
        j = int(j)
        z[:, c] = [O.keyed_normal(seed, sweep, purpose, j, i) for i in range(n)]
    return z


def draw_theta_rows(O, ts, y, prior, fstar, seed, sweep, rows):
    """O.draw_theta (mode 1) on respondents `rows` of y, addressed by their global indices; the rows are split over
    threads (every respondent is independent given f*, draw-theta.cpp:12-34, and the oracle releases the GIL)"""
    rows = np.asarray(rows)
    chunks = [c for c in np.array_split(rows, max(1, min(len(rows), os.cpu_count() or 1))) if c.size]

    def one(rr):
        rng = O.Rng.keyed(seed)
        rng.set_sweep(sweep)
        rng.set_respondent_map(rr)
        return O.draw_theta(ts, y[rr, :], prior, fstar, rng, mode=1)

    with ThreadPoolExecutor(len(chunks)) as ex:
        parts = list(ex.map(one, chunks))
    return (np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]),
            np.concatenate([p[2] for p in parts], axis=0))
