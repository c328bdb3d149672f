"""The compacted stream-K plan of the tile-skipping gather (csrc/gather.cu build_skip_plan / next_piece), checked on the host
through daisy_gather_plan_dump: no GPU needed."""
import ctypes as C

import numpy as np
import pytest


def _dump(occ, sms):
    from daisyriot_b200 import _lib
    L = _lib.lib()
    occ = np.ascontiguousarray(occ, np.uint8)
    nrb, S = occ.shape
    u8 = occ.ctypes.data_as(C.POINTER(C.c_uint8))
    info = np.zeros(5, np.int32)
    _lib.check(L.daisy_gather_plan_dump(u8, nrb, S, sms, _lib.iptr(info), None, None, None, 0))
    total, grid, Lmax, maxp, npieces = (int(v) for v in info)
    cap = max(total, nrb + 1, 6 * npieces, 1)
    lst, off, pcs = np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap, np.int32)
    _lib.check(L.daisy_gather_plan_dump(u8, nrb, S, sms, _lib.iptr(info), _lib.iptr(lst), _lib.iptr(off), _lib.iptr(pcs), cap))
    return (total, grid, Lmax, maxp), lst[:total], off[:nrb + 1], pcs[:6 * npieces].reshape(-1, 6)


def _maps():
    rng = np.random.RandomState(7)
    yield "random", (rng.uniform(size=(97, 33)) < 0.4)
    m = rng.uniform(size=(128, 64)) < 0.5
    m[10:40] = False          # whole zero row blocks
    m[:, 20:30] = False       # whole zero column steps
    yield "zero_blocks", m
    yield "all_zero", np.zeros((50, 17), bool)
    m = np.zeros((50, 17), bool)
    m[-1, -1] = True
    yield "last_tile_only", m
    yield "dense", np.ones((40, 9), bool)
    yield "one_row_block", rng.uniform(size=(1, 300)) < 0.3


@pytest.mark.parametrize("sms", [1, 7, 148])
def test_plan_covers_every_occupied_tile_once(sms):
    for name, occ in _maps():
        (total, grid, Lmax, maxp), lst, off, pcs = _dump(occ, sms)
        nrb, S = occ.shape
        # every row block has at least one entry; its entries are its occupied steps in order, or one null entry
        assert off[0] == 0 and off[-1] == total and np.all(np.diff(off) >= 1), name
        for rb in range(nrb):
            want = np.flatnonzero(occ[rb])
            got = lst[off[rb]:off[rb + 1]]
            assert np.array_equal(got, want) if want.size else (got.tolist() == [-1]), (name, rb)
        assert grid == min(sms, total), name
        # CTA ranges are contiguous, cover [0, total) exactly once, and differ in length by at most one
        lens = np.zeros(grid, np.int64)
        seen = np.zeros(total, np.int64)
        for c in range(grid):
            mine = pcs[pcs[:, 0] == c]
            assert mine.shape[0] >= 1, (name, c)
            pos = None
            for _, rb, e0, e1, idx, np_ in mine:
                assert off[rb] <= e0 <= e1 <= off[rb + 1], (name, c, rb)
                assert pos is None or e0 == pos, (name, c)
                # a null entry comes back as an empty range but still occupies its position
                end = e0 + 1 if (e1 == e0 and lst[e0] == -1) else e1
                assert end > e0, (name, c, rb)
                seen[e0:end] += 1
                lens[c] += end - e0
                pos = end
        assert np.all(seen == 1), name
        assert lens.max() - lens.min() <= 1 and lens.max() == Lmax, name
        # idx / np: the pieces of a row block in CTA order, as the plan's own ranges give them
        bounds = [c * total // grid for c in range(grid + 1)]
        for rb in range(nrb):
            ctas = [c for c in range(grid) if bounds[c] < off[rb + 1] and bounds[c + 1] > off[rb]]
            rows = pcs[pcs[:, 1] == rb]
            assert rows[:, 0].tolist() == ctas, (name, rb)
            assert rows[:, 4].tolist() == list(range(len(ctas))) and np.all(rows[:, 5] == len(ctas)), (name, rb)
            assert len(ctas) <= maxp
        # occupied tiles streamed = entries minus null entries
        assert int((lst >= 0).sum()) == int(occ.sum()), name


def test_plan_rejects_bad_arguments():
    from daisyriot_b200 import _lib
    info = np.zeros(5, np.int32)
    occ = np.ones((2, 2), np.uint8)
    u8 = occ.ctypes.data_as(C.POINTER(C.c_uint8))
    assert _lib.lib().daisy_gather_plan_dump(u8, 2, 2, 0, _lib.iptr(info), None, None, None, 0) != 0
    small = np.zeros(1, np.int32)
    assert _lib.lib().daisy_gather_plan_dump(u8, 2, 2, 4, _lib.iptr(info), _lib.iptr(small), None, None, 1) != 0
