# -*- coding: utf-8 -*-
"""N>1 host logic on CPU: the shard row ranges of george_b200.parallel.  The sharded factorisation itself needs GPUs
and the library's communicator (tools/mgpu_check.py and bench.py --gpus N)."""
import pytest


def test_shard_ranges():
    from george_b200.parallel import shard_ranges
    assert shard_ranges(1000, 1, 100) == [(0, 1000)]
    assert shard_ranges(1001, 2, 100) == [(0, 500), (500, 501)]
    assert shard_ranges(1001, 4, 100) == [(0, 250), (250, 250), (500, 250), (750, 251)]
    assert shard_ranges(300, 4, 100) is None
    with pytest.raises(ValueError):
        shard_ranges(100, 3, 10)
