"""-m "not gpu": the host-side planner of the symmetric self-search (csrc/nn_screen_tc.cu::plan_screen_sym) through
its test hook - no device work.  The multi-GPU scheme is only correct if the parts' triangle shares tile the upper
triangle EXACTLY ONCE; it is only fast if the shares are balanced and contiguous; the gated (upload-overlapped) order
only avoids waiting on itself if no unit needs a chunk later than its gate."""
import ctypes

import numpy as np
import pytest

from video_similarity_search_b200 import _lib

ROWS = 256   # rows of a unit (a CTA pair)
TILE = 256   # columns of a tile


def plan(n, part=0, parts=1, mode=0, gated_chunks=0):
    lib = _lib.load()
    num = ctypes.c_int64(0)
    _lib.check(lib.slic_debug_sym_plan(n, part, parts, mode, gated_chunks, None, 0, ctypes.addressof(num)), "plan")
    out = np.zeros((num.value, 6), dtype=np.int32)
    _lib.check(lib.slic_debug_sym_plan(n, part, parts, mode, gated_chunks, out.ctypes.data, num.value,
                                       ctypes.addressof(num)), "plan")
    return out


def upper_triangle(n):
    """want[r, ct] = 1 iff column tile ct lies on or right of row unit r's diagonal tile."""
    R, T = -(-n // ROWS), -(-n // TILE)
    return (np.arange(T)[None, :] >= np.arange(R)[:, None]).astype(np.int32)


def tiles_of(units):
    return [(int(r), int(c0 + k * st)) for r, c0, cnt, st, _, _ in units for k in range(cnt)]


@pytest.mark.parametrize("n,parts", [(16384, 1), (16384, 2), (41003, 3), (240000, 8), (240000, 5), (1000000, 8)])
def test_triangle_shares_tile_the_upper_triangle_exactly_once(n, parts):
    want = upper_triangle(n)
    seen = np.zeros_like(want)
    share = []
    for mode in (2, 3):                                                  # the triangle alone / behind the fused pre-pass
        seen[:] = 0
        share = []
        for part in range(parts):
            u = plan(n, part, parts, mode=mode)
            u = u[u[:, 5] == 1]
            assert (u[:, 4] == -1).all()                                 # triangle units, ungated
            t = np.array(tiles_of(u))
            np.add.at(seen, (t[:, 0], t[:, 1]), 1)
            share.append(len(t))
        assert np.array_equal(seen, want)                                # every tile on or right of the diagonal, once
        assert sum(share) == int(want.sum())
        assert max(share) - min(share) <= 2 * 64                         # balanced to a unit (<= 16 384 columns) either way


def test_full_mode_is_prepass_plus_the_same_triangle_and_row_bests_cover_every_row_once():
    n, parts = 240000, 8
    R, T = -(-n // ROWS), -(-n // TILE)
    rows, fused_rows = [], []
    for part in range(parts):
        full, tri, pre = plan(n, part, parts, 0), plan(n, part, parts, 2), plan(n, part, parts, 1)
        assert np.array_equal(full[full[:, 5] == 1], tri)                # mode 0 = pre-pass over all rows + this share
        assert sorted(full[full[:, 5] == 0][:, 0].tolist()) == list(range(R))
        assert (pre[:, 5] == 0).all() and (pre[:, 2] == 32).all()        # 32 x 256 sampled columns from 4 parts on
        cols = np.array([c for _, c in tiles_of(pre[:1])])
        assert cols.min() >= 0 and cols.max() < T and len(set(cols.tolist())) == 32
        rows += pre[:, 0].tolist()
        # fused (multi-GPU kernel): the same rows and the same sample, cut into units of 16 x 256 columns, then the share
        fused = plan(n, part, parts, 3)
        fpre = fused[fused[:, 5] == 0]
        assert np.array_equal(fused[fused[:, 5] == 1], tri) and (np.diff(fused[:, 5]) >= 0).all()
        assert (fpre[:, 2] == 16).all() and len(fpre) == 2 * len(pre)
        assert sorted(tiles_of(fpre)) == sorted(tiles_of(pre))
        fused_rows += sorted(set(fpre[:, 0].tolist()))
    assert sorted(rows) == list(range(R)) and sorted(fused_rows) == list(range(R))   # every row block on exactly one part
    assert (plan(n, 0, 2, 1)[:, 2] == 16).all()                          # 16 x 256 columns below 4 parts
    small = plan(16384, 0, 8, 1)                                         # 64 x 256 columns in all: a quarter is sampled
    assert (small[:, 2] == 16).all()


@pytest.mark.parametrize("n,chunks", [(80000, 4), (240000, 8), (100003, 8), (32768, 8)])
def test_gated_order_never_needs_a_chunk_later_than_its_gate(n, chunks):
    u = plan(n, 0, 1, 0, gated_chunks=chunks)
    chunk_rows = -(-(-(-n // chunks)) // ROWS) * ROWS
    tiles_per_chunk, units_per_chunk = chunk_rows // TILE, chunk_rows // ROWS
    gates = u[:, 4]
    assert (gates >= 0).all() and (np.diff(gates) >= 0).all()            # consumed in arrival order
    for r, c0, cnt, st, g, cdir in u:
        last_col = c0 + (cnt - 1) * st
        assert g >= r // units_per_chunk and g >= last_col // tiles_per_chunk
    # inside a gate the pre-pass units come before the triangle units that wait for their thresholds
    for g in np.unique(gates):
        flags = u[gates == g][:, 5]
        assert (np.diff(flags) >= 0).all()
    want = upper_triangle(n)
    seen = np.zeros_like(want)
    t = np.array(tiles_of(u[u[:, 5] == 1]))
    np.add.at(seen, (t[:, 0], t[:, 1]), 1)
    assert np.array_equal(seen, want)
