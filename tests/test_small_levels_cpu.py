"""CPU: hashgrid._field.small_levels -- the count of single-pass coarse levels that decides the slicing plan of the fused
scatter + Adam backward is cached per resolution tensor; a different tensor at the same address, or the same tensor changed
in place, must be counted again (the plan would otherwise follow a ladder that is no longer there)."""
import numpy as np
import torch

from conftest import load_pkg
from oracle import torch_ref as tr

C2 = tr.resolution_ladder(torch.tensor([49, 32, 73]), torch.tensor([12603, 8192, 18904])).int()     # BASELINE.json C2
FINE = tr.resolution_ladder(torch.tensor([16, 16, 16]), torch.tensor([4096, 4096, 4096])).int()


def test_in_place_change_is_counted_again():
    load_pkg()
    from hashgrid import _field
    a = C2.clone()
    assert _field.small_levels(a) == 4
    assert _field.small_levels(a) == 4          # cached
    a.copy_(FINE)
    assert _field.small_levels(a) == 7
    a[:] = C2
    assert _field.small_levels(a) == 4


def test_new_tensor_at_the_old_address_is_counted_again():
    load_pkg()
    from hashgrid import _field
    buf = C2.numpy().copy()
    a = torch.from_numpy(buf)
    ptr = a.data_ptr()
    assert _field.small_levels(a) == 4
    del a
    buf[...] = FINE.numpy()                     # the memory is reused for another ladder, written outside torch
    b = torch.from_numpy(buf)
    assert b.data_ptr() == ptr and b.shape == C2.shape
    assert _field.small_levels(b) == 7


def test_cache_entry_dies_with_its_tensor():
    load_pkg()
    from hashgrid import _field
    a = torch.from_numpy(np.ascontiguousarray(C2.numpy()))
    _field.small_levels(a)
    assert a in _field._small_levels_cache
    n = len(_field._small_levels_cache)
    del a
    assert len(_field._small_levels_cache) == n - 1
