"""Property tests (hypothesis) of the host-side logic: the DCN tile plan and the ragged-batch sharding.  CPU only."""
import ctypes

import numpy as np
from hypothesis import given, settings, strategies as st

from mrefsr_b200 import _lib, parallel as P


@settings(max_examples=80, deadline=None)
@given(b=st.integers(1, 5), ho=st.integers(1, 70), wo=st.integers(1, 70))
def test_tile_plan_is_a_bijection_onto_the_output_positions(b, ho, wo):
    lib = _lib.lib()
    meta = (ctypes.c_int * 4)()
    assert lib.mrefsr_dcn_tile_plan(b, ho, wo, ctypes.cast(meta, ctypes.c_void_p), None, 0) == 0
    tile2d, pw, ph, tiles = list(meta)
    lin_tiles = -(-b * ho * wo // 256)
    assert lin_tiles <= tiles and tiles * 100 <= lin_tiles * 103
    coords = np.full((tiles * 256, 3), -7, dtype=np.int32)
    assert lib.mrefsr_dcn_tile_plan(b, ho, wo, ctypes.cast(meta, ctypes.c_void_p), coords.ctypes.data_as(ctypes.c_void_p),
                                    tiles * 256) == 0
    valid = coords[:, 0] >= 0
    assert (coords[~valid] == -1).all()
    c = coords[valid].astype(np.int64)
    assert (c[:, 0] < b).all() and (c[:, 1] < ho).all() and (c[:, 2] < wo).all() and (c[:, 1:] >= 0).all()
    lin = (c[:, 0] * ho + c[:, 1]) * wo + c[:, 2]
    assert len(lin) == b * ho * wo == len(np.unique(lin))
    if tile2d:
        # every patch lies inside one sample and spans at most pw x ph positions
        per = pw * ph
        for k in range(0, len(coords), per):
            blk = coords[k:k + per]
            blk = blk[blk[:, 0] >= 0]
            if len(blk):
                assert (blk[:, 0] == blk[0, 0]).all()
                assert blk[:, 1].max() - blk[:, 1].min() < ph and blk[:, 2].max() - blk[:, 2].min() < pw


@settings(max_examples=100, deadline=None)
@given(counts=st.lists(st.integers(1, 8), min_size=0, max_size=40), world=st.integers(1, 9))
def test_shard_ragged_partitions_and_respects_the_lpt_bound(counts, world):
    owned = P.shard_ragged(counts, world)
    assert len(owned) == world and sorted(sum(owned, [])) == list(range(len(counts)))
    loads = [sum(P.image_cost(counts[i]) for i in o) for o in owned]
    if counts:
        assert max(loads) - min(loads) <= max(P.image_cost(c) for c in counts) + 1e-9
    for r in range(world):
        assert P.shard_ragged(counts, world, r) == owned[r]


@settings(max_examples=100, deadline=None)
@given(keys=st.lists(st.integers(0, 4), min_size=0, max_size=60), max_batch=st.integers(1, 7))
def test_batches_by_shape_is_an_order_preserving_partition(keys, max_batch):
    got = P.batches_by_shape(keys, max_batch)
    flat = [i for _, idxs in got for i in idxs]
    assert sorted(flat) == list(range(len(keys)))
    for k, idxs in got:
        assert 1 <= len(idxs) <= max_batch and idxs == sorted(idxs) and all(keys[i] == k for i in idxs)
    # buckets of one key are filled in order: only the last bucket of a key may be short
    for k in set(keys):
        sizes = [len(idxs) for kk, idxs in got if kk == k]
        assert all(s == max_batch for s in sizes[:-1])

