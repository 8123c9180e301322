"""CPU (-m "not gpu"): the engine's slot pipeline against a fake library -- submits go round the slots, waits come in submit
order (the oldest before its slot is reused), every tile is waited for, and an input of no sites is one empty tile."""
import numpy as np
import pytest

from basevar_b200 import capi
from basevar_b200.engine import BaseTypeEngine


class FakeLib:
    def __init__(self):
        self.log = []

    def bv_tile_submit(self, ctx, slot, tile):
        self.log.append(("submit", slot, tile._obj.n_sites))
        return capi.BV_OK

    def bv_tile_wait(self, ctx, slot, out):
        self.log.append(("wait", slot))
        return capi.BV_OK


def fake_engine(n_slots, max_sites):
    eng = BaseTypeEngine.__new__(BaseTypeEngine)
    eng.lib, eng._ctx = FakeLib(), None
    eng.params = capi.make_params(max_samples=16, max_sites=max_sites, n_slots=n_slots)
    return eng


def run(n_slots, n_sites, max_sites=2):
    eng = fake_engine(n_slots, max_sites)
    planes = [np.zeros((n_sites, 16), np.uint8) for _ in range(3)]
    eng.call_host(*planes, np.zeros(n_sites, np.uint8), 16)
    return eng.lib.log


def test_one_slot_waits_after_every_submit():
    assert run(1, 5) == [("submit", 0, 2), ("wait", 0), ("submit", 0, 2), ("wait", 0), ("submit", 0, 1), ("wait", 0)]


def test_three_slots_wait_fifo():
    assert run(3, 9) == [("submit", 0, 2), ("submit", 1, 2), ("submit", 2, 2),
                         ("wait", 0), ("submit", 0, 2), ("wait", 1), ("submit", 1, 1),
                         ("wait", 2), ("wait", 0), ("wait", 1)]


@pytest.mark.parametrize("n_slots", [1, 3])
def test_no_sites_is_one_empty_tile(n_slots):
    assert run(n_slots, 0) == [("submit", 0, 0), ("wait", 0)]
