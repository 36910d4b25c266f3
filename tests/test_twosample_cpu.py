"""The two-sample test without a GPU: mmd_from_sums against a direct double loop, the p-value
rule, NaN groups, KS D against scipy, bf16 features, the definition of two_sample_test on
mocked components (groups, subsample and labelling draws, the network's RNG streams), the CSV
writer and the `twosample` command's argument and file checks."""
import os
from unittest.mock import MagicMock

import numpy as np
import pytest
import scipy.stats

from cellcomm_b200.bigan_basic import (BasicBiGan, MMD_SCALES, TwoSampleTest, bf16_round,
                                       kernel_sums, ks_statistic, log1p_features,
                                       mmd_from_sums, pack_labellings, permutation_p_value,
                                       two_sample_cells, two_sample_labellings)


def _direct(k, x):
    """fp64 double loop over ordered pairs i != j of the kernel matrix k, X = the cells in x"""
    N = len(k)
    xx = yy = xy = 0.0
    for i in range(N):
        for j in range(N):
            if i == j:
                continue
            if x[i] and x[j]:
                xx += k[i, j]
            elif not x[i] and not x[j]:
                yy += k[i, j]
            elif x[i]:
                xy += k[i, j]
    return xx, yy, xy


def test_mmd_from_sums_and_kernel_sums_match_a_double_loop():
    rng = np.random.default_rng(0)
    F = rng.normal(size=(14, 5))
    G = F @ F.T
    g = np.diag(G)
    d2 = np.maximum(g[:, None] + g[None, :] - 2 * G, 0)
    masks = two_sample_labellings(7, 6, 3, 0)
    sums = kernel_sums(d2, masks, [1.0, 4.0])
    for p, x in enumerate(masks):
        for b, h in enumerate([1.0, 4.0]):
            want = _direct(np.exp(-d2 / h), x)
            np.testing.assert_allclose(sums[p, b], want, rtol=1e-12)
            xx, yy, xy = want
            n = 7
            mmd = 0.0
            # the textbook form: mean over i != j in X, in Y, minus twice the mean over X x Y
            mmd = xx / (n * (n - 1)) + yy / (n * (n - 1)) - 2 * xy / (n * n)
            assert mmd_from_sums(n, *sums[p, b]) == pytest.approx(mmd, rel=1e-12)


def test_p_value_rule():
    stats = np.array([[0.5, 0.1], [0.5, 0.2], [0.4, 0.0], [0.6, 0.3]])
    np.testing.assert_array_equal(permutation_p_value(stats), [3 / 4, 3 / 4])
    assert permutation_p_value(np.array([[1.0]]))[0] == 1.0          # no permutation


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_ks_matches_scipy(seed):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 20, 300).astype(np.float64)                    # ties
    b = rng.integers(3, 25, 211).astype(np.float64)
    assert ks_statistic(a, b) == pytest.approx(scipy.stats.ks_2samp(a, b).statistic, abs=1e-15)
    c = rng.normal(size=50)
    assert ks_statistic(c, c) == 0.0
    assert np.isnan(ks_statistic([], c))


def test_bf16_features():
    import torch
    v = np.array([0.0, -0.0, 1.0, 3.0, 255.0, 256.0, 1e6, 0.5, np.nan], np.float64)
    f = log1p_features(v)
    want = torch.tensor(np.log1p(v).astype(np.float32)).to(torch.bfloat16).float().numpy()
    np.testing.assert_array_equal(f[:-1], want[:-1])
    assert np.signbit(f[1]) and not np.signbit(f[0])
    assert np.isnan(f[-1])
    x = np.random.default_rng(1).normal(size=10000).astype(np.float32) * 100
    np.testing.assert_array_equal(bf16_round(x), torch.tensor(x).to(torch.bfloat16).float().numpy())


def test_labellings_and_packing():
    m = two_sample_labellings(5, 4, 9, 2)
    assert m.shape == (5, 10) and (m.sum(1) == 5).all() and m[0, :5].all()
    rng = np.random.default_rng([9, 1, 2])
    for p in range(1, 5):
        assert set(np.flatnonzero(m[p])) == set(rng.permutation(10)[:5])
    packed = pack_labellings(np.eye(40, dtype=bool)[:3])
    assert packed.dtype == np.uint32 and packed.shape == (3, 2)
    np.testing.assert_array_equal(packed, [[1, 0], [2, 0], [4, 0]])
    assert pack_labellings(np.eye(40, dtype=bool)[33:34])[0, 1] == 2


def test_subsample_draw():
    labels = np.array([0, 1, 0, 0, 1, 0, 0, 2])
    picks = two_sample_cells(labels, 4, 3, 11)
    rows0 = np.flatnonzero(labels == 0)
    want = rows0[np.sort(np.random.default_rng([11, 0, 0]).choice(5, 3, replace=False))]
    np.testing.assert_array_equal(picks[0], want)
    np.testing.assert_array_equal(picks[1], [1, 4])
    np.testing.assert_array_equal(picks[2], [7])
    assert len(picks[3]) == 0


# ------------------------------------------------------------------ the definition on mocks
class _Basic(BasicBiGan):
    def random_encoding_vector(self, n):
        return self._prior_rng.random((n, self.encoding_size), dtype=np.float32)

    def trainings_step(self, batch):
        pass


def _generate(inputs):
    z, r = (np.asarray(a, dtype=np.float32) for a in inputs)
    base = np.arange(6, dtype=np.float32)
    return (base[None, :] * (1 + 2 * z[:, :1]) + 4 * r[:, :1]).astype(np.float32)


def _mocked(Z=2, G=6):
    comps = [MagicMock() for _ in range(3)]
    comps[0].predict = MagicMock(side_effect=_generate)
    net = _Basic(Z, G, *(MagicMock(return_value=c) for c in comps))
    net._prior_rng = np.random.default_rng(5)
    return net, comps


def _reference(net_state, x, labels, K, max_cells, P, seed, net):
    """the definition spelled out step by step"""
    picks = two_sample_cells(labels, K, max_cells, seed)
    net._prior_rng.bit_generator.state = net_state
    enc = net._comparison_encodings([len(p) for p in picks])
    noise = net.random_uniform_vector(len(enc))
    gen = np.round(_generate((enc, noise))).astype(np.float64)
    out, off = [], 0
    for k in range(K):
        n = len(picks[k])
        F = np.concatenate([log1p_features(x[picks[k]]), log1p_features(gen[off:off + n])])
        F = F.astype(np.float64)
        G = F @ F.T
        g = np.diag(G)
        d2 = np.maximum(g[:, None] + g[None, :] - 2 * G, 0)
        med = np.sort(d2[np.triu_indices(2 * n, 1)])[(n * (2 * n - 1) - 1) // 2]
        stats = []
        for x_mask in two_sample_labellings(n, P, seed, k):
            row = []
            for s in MMD_SCALES:
                row.append(mmd_from_sums(n, *_direct(np.exp(-d2 / (s * med)), x_mask)))
            stats.append(row)
        stats = np.array(stats)
        out.append((med, stats[0], permutation_p_value(stats),
                    ks_statistic(x[picks[k]].sum(1), gen[off:off + n].sum(1))))
        off += n
    return out


def test_definition_on_mocks():
    net, comps = _mocked()
    x = np.random.default_rng(3).integers(0, 4, (11, 6)).astype(np.float64)
    state = net._prior_rng.bit_generator.state
    np_state = np.random.get_state()
    t = net.two_sample_test(x, max_cells=8, permutations=9, seed=4)
    assert isinstance(t, TwoSampleTest)
    assert np.random.get_state()[1].tobytes() == np_state[1].tobytes()
    after = net._prior_rng.bit_generator.state
    # the network's stream moved by exactly what compare_cells would draw for 8 cells
    net._prior_rng.bit_generator.state = state
    net._comparison_encodings([8])
    net.random_uniform_vector(8)
    assert net._prior_rng.bit_generator.state == after
    np.testing.assert_array_equal(t.real_cells, [8])
    np.testing.assert_array_equal(t.generated_cells, [8])
    (med, mmd, p, ks), = _reference(state, x, np.zeros(11, np.int64), 1, 8, 9, 4, net)
    assert t.sqdist_median[0] == med
    np.testing.assert_allclose(t.mmd2[0], mmd, rtol=1e-9, atol=1e-12)
    np.testing.assert_array_equal(t.p_value[0], p)
    assert t.library_size_ks[0] == ks
    assert t.mmd2.shape == (1, 3) and t.p_value.dtype == np.float64


def test_groups_and_nan_groups():
    net, _ = _mocked()
    net._comparison_groups = lambda cells: (np.array([0, 0, 0, 2, 0, 0]), 3)
    x = np.random.default_rng(4).integers(0, 5, (6, 6)).astype(np.float64)
    t = net.two_sample_test(x, permutations=5)
    np.testing.assert_array_equal(t.real_cells, [5, 0, 1])
    assert not np.isnan(t.mmd2[0]).any()
    for k in (1, 2):
        assert np.isnan(t.mmd2[k]).all() and np.isnan(t.p_value[k]).all()
        assert np.isnan(t.sqdist_median[k]) and np.isnan(t.library_size_ks[k])
    # all cells identical: the median is 0 and there is no test
    same = np.ones((6, 6))
    net2, _ = _mocked()
    net2._generator.predict = MagicMock(return_value=np.ones((6, 6), np.float32))
    t2 = net2.two_sample_test(same, permutations=3)
    assert t2.sqdist_median[0] == 0.0 and np.isnan(t2.mmd2).all()


def test_argument_checks():
    net, _ = _mocked()
    x = np.ones((4, 6))
    for kw in ({"max_cells": 1}, {"max_cells": 16385}, {"permutations": -1}, {"seed": -2}):
        with pytest.raises(ValueError):
            net.two_sample_test(x, **kw)
    with pytest.raises(ValueError, match="negative"):
        net.two_sample_test(-x)


# ------------------------------------------------------------------ the CSV and the command
def test_csv_writer(tmp_path):
    from cellcomm_b200.__main__ import TWOSAMPLE_COLUMNS, write_twosample_file
    t = TwoSampleTest(np.array([5, 1]), np.array([5, 1]), np.array([0.1, np.nan]),
                      np.array([[1e-3, 2e-3, 3e-3], [np.nan] * 3]),
                      np.array([[0.5, 0.25, 1 / 3], [np.nan] * 3]),
                      np.array([0.2, np.nan]), np.array([0.4, np.nan]))
    path = write_twosample_file(str(tmp_path / "t.csv"), t)
    lines = open(path).read().splitlines()
    assert lines[0] == ",".join(TWOSAMPLE_COLUMNS)
    assert lines[0] == ("group,real-cells,generated-cells,sqdist-median,mmd2-s0.5,p-s0.5,"
                        "mmd2-s1,p-s1,mmd2-s2,p-s2,library-size-ks,genes-detected-ks")
    f = lines[1].split(",")
    assert f[:3] == ["0", "5", "5"]
    assert [float(v) for v in f[3:]] == [0.1, 1e-3, 0.5, 2e-3, 0.25, 3e-3, 1 / 3, 0.2, 0.4]
    assert lines[2].startswith("1,1,1,nan,")
    assert sorted(os.listdir(tmp_path)) == ["t.csv"]


def test_command_checks_arguments_and_files(tmp_path):
    from cellcomm_b200 import __main__ as cli
    with pytest.raises(AssertionError, match="twosample <checkpoint.npz>"):
        cli.main(["", "twosample", "a", "b"])
    built = MagicMock(side_effect=AssertionError("a network was built"))
    cli_restore = cli._restore_network
    cli._restore_network = built
    try:
        with pytest.raises(FileNotFoundError, match="no such file"):
            cli.main(["", "twosample", str(tmp_path / "none.npz"), str(tmp_path / "m.mtx"),
                      str(tmp_path / "c.mtx"), str(tmp_path / "o.csv")])
    finally:
        cli._restore_network = cli_restore
    assert not os.path.exists(tmp_path / "o.csv")
    assert "twosample" in cli.__doc__
