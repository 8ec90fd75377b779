"""CPU checks of subset stepping: the C entry points refuse a null handle, and the subset validator
(`batched_env.check_subset`) refuses empty, duplicate, out-of-range and non-integer ids and empty or
out-of-bounds ranges."""
import numpy as np
import pytest
import torch

from paintrl_b200.batched_env import check_subset


def test_subset_entry_points_refuse_a_null_handle():
    from paintrl_b200 import build
    build.build()
    from paintrl_b200 import _capi
    lib = _capi.lib()
    assert lib.paintrl_step_subset(None, None, 0, 4, *([None] * 10)) == -1
    assert b'null' in lib.paintrl_last_error()
    assert lib.paintrl_step_host_submit_range(None, 0, 0, 4, *([None] * 8)) == -1
    assert b'null' in lib.paintrl_last_error()


@pytest.mark.parametrize('bad, exc', [
    ([], ValueError),
    (np.array([], dtype=np.int64), ValueError),
    ([3, 3], ValueError),
    ([0, 5, 2, 5], ValueError),
    ([8], IndexError),
    ([-1, 2], IndexError),
    ([0.0, 1.0], ValueError),
    (np.array([True, False]), ValueError),
    (torch.tensor([1, 1]), ValueError),
    (range(0), ValueError),
    (range(4, 4), ValueError),
    (range(0, 8, 2), ValueError),
    (range(-1, 3), IndexError),
    (range(5, 9), IndexError),
])
def test_subset_validator_rejects(bad, exc):
    with pytest.raises(exc):
        check_subset(bad, 8)


def test_subset_validator_accepts():
    assert check_subset(range(2, 7), 8) == (None, 2, 5)
    assert check_subset(range(0, 8), 8) == (None, 0, 8)
    ids, lo, n = check_subset([7, 0, 3], 8)
    assert ids.dtype == np.int32 and ids.tolist() == [7, 0, 3] and (lo, n) == (0, 3)
    ids, lo, n = check_subset(torch.tensor([5, 1], dtype=torch.int64), 8)
    assert ids.tolist() == [5, 1] and n == 2
    ids, lo, n = check_subset(np.array([4], dtype=np.uint8), 8)
    assert ids.tolist() == [4] and n == 1
