"""The strata of tests/bench_strata.py cover every tile at the benchmark shapes (no GPU needed)."""
import numpy as np
import pytest

import bench_strata as B
from gpirt_b200 import synthetic


@pytest.mark.parametrize("workload,missing", [("c3", 0.0), ("c3", 0.05), ("c5", 0.0), ("c5", 0.05)])
def test_strata_cover_every_tile_and_upload_piece(workload, missing):
    c = synthetic.WORKLOADS[workload]
    n, m = c["n"], c["m"]
    big = n > 4096
    J, I = B.items(m, big), B.respondents(n, big)
    for name, idx, size, tile in (("items", J, m, B.DG_BN), ("respondents", I, n, B.TI_BM)):
        assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] == size - 1, name
        tiles = -(-size // tile)
        assert set(idx // tile) == set(range(tiles)), "%s: a %d-wide tile without a chosen index" % (name, tile)
        if not big:   # both ends of every tile, the ragged last one included
            assert len(idx) == 2 * tiles and set(idx) >= {t * tile for t in range(tiles)} | {size - 1}, name
    hit, pieces = B.upload_pieces(n, m, J)
    assert hit == set(range(pieces)), "an upload piece of y without a chosen item (%g missing)" % missing
    # the sizes the oracle tests are costed for: C3 2 x 157 items and 2 x 32 respondents; C5 313 + 1 items and 128
    # respondents (the alternation ends on the last row of the last tile, n - 1)
    assert (len(J), len(I)) == ((314, 64) if workload == "c3" else (314, 128))
    assert pieces == (10 if workload == "c3" else 79)
    assert len(B.panel_rows(n)) == 2 * n // B.CHOL_NB


def test_strata_on_ragged_and_single_tiles():
    assert list(B.tile_strata(130, 64, True)) == [0, 63, 64, 127, 128, 129]
    assert list(B.tile_strata(130, 64, False)) == [0, 127, 128, 129]
    assert list(B.tile_strata(1, 64, True)) == [0] and list(B.tile_strata(1, 64, False)) == [0]
    hit, pieces = B.upload_pieces(4096, 10000, [1023, 1024])
    assert pieces == 10 and hit == {0, 1}
