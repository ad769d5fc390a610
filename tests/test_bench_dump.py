"""bench.py --dump-outputs: what it writes for each workload, without a GPU.  The library handle is replaced by a stand-in with
accumulator slots: it starts as the timed light cone leaves them (the last two groups in their slot ranges) and answers fetch with
maps and counts that depend on the group in the slot, so a plane dumped under the wrong group shows."""
import functools
import os
import types

import numpy as np
import pytest

import bench

L = bench.LENS_PER_SNAP


@functools.lru_cache(maxsize=None)
def base_map(npix):
    return (np.arange(npix * npix) % 10007).astype(np.float32)


def planes_of(g, k, ptype, npix):
    m = base_map(npix) + np.float32(97 * g + 13 * k + ptype + 11)
    return m, np.arange(6, dtype=np.int64) * (g + 1) + k, np.full(6, g, np.int64)


class SlotStub:
    def __init__(self, ngroups):
        self.in_slot = {}
        for g in (ngroups - 2, ngroups - 1):
            for k in range(L):
                self.in_slot[(g & 1) * L + k] = (g, k)
        self.deposits = []

    def deposit_slots(self, group, first_slot):  # `group`: the stand-in's plane list is the group index
        self.deposits.append(group)
        for k in range(L):
            self.in_slot[first_slot + k] = (group, k)

    def settle_slots(self, first_slot, n):
        pass

    def fetch(self, slot, ptype, npix):
        g, k = self.in_slot[slot]
        m, c, i = planes_of(g, k, ptype, npix)
        return m.reshape(npix, npix), c, i


@pytest.mark.parametrize("name", sorted(bench.WORKLOADS))
def test_dump_covers_every_group_sampled_and_under_64_mb(tmp_path, name):
    W = bench.WORKLOADS[name]
    ngr, npix = W["ngroups"], W["npix"]
    stub = SlotStub(ngr)
    bench.dump_outputs(types.SimpleNamespace(W=W, s=stub, groups=list(range(ngr))), str(tmp_path))
    assert stub.deposits == list(range(ngr - 2))  # only the groups the step overwrote are deposited again
    files = sorted(os.listdir(tmp_path))
    assert sum(os.path.getsize(tmp_path / f) for f in files) < 64e6
    arrs = {f[:-4]: np.load(tmp_path / f) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in arrs.values())
    idx = arrs["pixel_index"].astype(np.int64)  # every workload's maps exceed the budget: one sample for all of them
    assert np.all(np.diff(idx) > 0) and idx[-1] < npix * npix
    ptypes = [0, 1, 4] if W["per_type"] else [-1]
    for g in range(ngr):
        for k in range(L):
            _, c, i = planes_of(g, k, ptypes[0], npix)
            assert arrs[f"group{g}_counts"][k].tolist() == c.tolist() and arrs[f"group{g}_ingrid"][k].tolist() == i.tolist()
            for t in ptypes:
                key = f"group{g}_maps" + (f"_type{t}" if t >= 0 else "")
                full = planes_of(g, k, t, npix)[0]
                assert np.array_equal(arrs[key][k], full[idx])
                assert arrs[key.replace("maps", "map_sums")][k] == full.sum(dtype=np.float64)
    assert len(files) == 1 + ngr * (2 + 2 * len(ptypes))
