"""tests/peer_ref.py, the host reference of tests/test_peer_exact_gpu.py, without a GPU."""
import numpy as np
import pytest

import peer_ref as P

F32 = np.float32


def bits(x):
    return np.asarray(x, F32).view(np.uint32)


def test_rank_order_sum_is_sequential_fp32_from_plus_zero():
    rng = np.random.default_rng(1)
    t = rng.standard_normal((5, 1000)).astype(F32)
    want = np.zeros(1000, F32)
    for q in range(5):
        want = (want + t[q]).astype(F32)
    assert np.array_equal(bits(P.rank_order_sum(t)), bits(want))
    # every term -0.0: the +0.0 start makes the sum +0.0
    assert bits(P.rank_order_sum(np.full((3, 2), -0.0, F32))).tolist() == [0, 0]
    assert bits(P.rank_order_sum(t[:1])).tolist() == bits(t[0]).tolist()


def test_hand_worked_order_case():
    """(1, 0.75 * 2^-24, -1): forward the small term is lost above 1 and the sum is 0; reversed
    -1 + 0.75 * 2^-24 rounds to -(1 - 2^-24) (the spacing halves below 1), so the sum is 2^-24."""
    t = np.array([[1.0], [0.75 * 2.0 ** -24], [-1.0]], F32)
    assert P.rank_order_sum(t)[0] == 0.0
    assert P.reverse_order_sum(t)[0] == F32(2.0 ** -24)
    assert P.pairwise_sum(t)[0] == 0.0                   # ((g0 + g1) + g2): the forward order
    t4 = np.array([[1.0], [0.75 * 2.0 ** -24], [-1.0], [3.0 * 2.0 ** -30]], F32)
    assert P.pairwise_sum(t4)[0] != P.rank_order_sum(t4)[0]


@pytest.mark.parametrize("world", [1, 2, 3, 4, 5, 8, 16])
def test_order_terms_make_the_order_observable(world):
    rng = np.random.default_rng(world)
    g, mask = P.order_terms(rng, world, 20000)
    assert g.dtype == F32 and g.shape == (world, 20000)
    fwd, rev = P.rank_order_sum(g), P.reverse_order_sum(g)
    if world < 3:
        assert not mask.any()
        assert np.array_equal(bits(fwd), bits(rev))      # fp32 addition of two terms commutes
        return
    assert 0.4 < mask.mean() < 0.6
    assert np.mean(bits(fwd)[mask] != bits(rev)[mask]) > 0.99
    if world >= 4:
        assert np.mean(bits(fwd)[mask] != bits(P.pairwise_sum(g))[mask]) > 0.9
    assert np.all(np.isfinite(fwd))
    # the forward sum of the order elements is the sum of the fine terms alone
    fine = P.rank_order_sum(g[3:, mask]) if world > 3 else np.zeros(mask.sum(), F32)
    assert np.array_equal(bits(fwd[mask]), bits(np.float32(0) + fine))


def test_zero_and_negative_zero_elements():
    g, _ = P.order_terms(np.random.default_rng(0), 4, 1000)
    assert np.all(bits(g[:, 3::23]) == 0)
    negz = bits(g[:, 5::46]) == 0x80000000
    assert negz.all(axis=0).any()


def test_epoch_arithmetic_is_modular():
    assert P.effective_epoch(5) == 5
    assert P.effective_epoch(1, 2 ** 32 - 2) == 2 ** 32 - 1
    assert P.effective_epoch(1, 2 ** 32 - 1) == 0
    assert P.effective_epoch(3, 2 ** 32 - 1) == 2
    assert P.effective_epoch(1, -1) == 0                 # a counter read back as int32
    for v in (0, 1, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1):
        assert P.u32(P.as_i32(v)) == v
        assert -2 ** 31 <= P.as_i32(v) < 2 ** 31
    assert P.as_i32(2 ** 32 - 1) == -1


def test_flag_comparison_matches_wait_flag():
    assert P.flag_reached(5, 5) and P.flag_reached(6, 5)
    assert not P.flag_reached(4, 5)
    assert P.flag_reached(0, 2 ** 32 - 1)                # the flag has wrapped past the epoch
    assert not P.flag_reached(2 ** 32 - 1, 0)
    assert P.flag_reached(7 + 2 ** 31 - 1, 7)
    assert not P.flag_reached(7 + 2 ** 31, 7)
    assert P.flag_reached(-1, 2 ** 32 - 1)               # int32 flag storage


def test_allreduce_slot_addressing():
    W, cap = 5, 33
    seen = set()
    for e in (6, 7):
        for src in range(W):
            o = P.ar_slot_offset(e, W, cap, src)
            assert o % cap == 0 and 0 <= o < 2 * W * cap
            seen.add(o)
    assert seen == {k * cap for k in range(2 * W)}       # disjoint slots cover the array
    assert P.ar_slot_offset(2 ** 32 - 1, W, cap, 0) == W * cap
    assert P.ar_slot_offset(0, W, cap, 0) == 0           # parity flips across the wrap
    assert [P.ar_parity(e) for e in (1, 2, 3)] == [1, 0, 1]
    assert [P.ar_threads(n) for n in (1, 31, 32, 33, 1023, 1024, 1025)] == \
        [32, 32, 32, 64, 1024, 1024, 1024]


def test_launch_geometry():
    assert P.blocks_per_sm(None) == 2
    assert [P.blocks_per_sm(v) for v in ("1", "8", "4", " 3", "3x", "0", "9", "-1", "", "x")] == \
        [1, 8, 4, 3, 3, 2, 2, 2, 2, 2]
    sms, per = 148, 2
    assert P.rmsprop_passes(0, sms, per) == 0
    assert P.rmsprop_passes(8, sms, per) == 1 and P.rmsprop_grid(8, sms, per) == 1
    full = 8 * 256 * sms * per
    assert P.rmsprop_passes(full, sms, per) == 1
    assert P.rmsprop_passes(full + 8, sms, per) == 2
    assert P.rmsprop_grid(10 * full, sms, per) == sms * per


def test_lo_mask_uses_the_group_start():
    off = np.arange(64, 128)
    m = P.lo_mask(off, [(80, 96), (120, 120)])
    assert m.tolist() == [(80 <= o < 96) for o in range(64, 128)]
    assert not P.lo_mask(off, []).any()
