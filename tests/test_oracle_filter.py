"""The filter oracle checks itself (CPU): batch pushes merged at sync time give the same statistics as RLlib-style
sequential Welford pushes, and both filters normalise as (x - mean) / (std + 1e-8) with clipping, the mean subtracted
only if demean and the std divided out only if destd."""
import numpy as np
import pytest

from oracle.filter_oracle import BatchSyncFilter, RunningStat, SequentialFilter


def test_running_stat_is_mean_and_unbiased_variance():
    rng = np.random.default_rng(0)
    x = rng.normal(3.0, 2.0, size=(500, 7))
    rs = RunningStat(7)
    for row in x:
        rs.push(row)
    np.testing.assert_allclose(rs.M, x.mean(0), rtol=1e-12)
    np.testing.assert_allclose(rs.var, x.var(0, ddof=1), rtol=1e-12)
    one = RunningStat(2)
    one.push([3.0, -2.0])
    np.testing.assert_allclose(one.var, [9.0, 4.0])          # n == 1: var reports mean^2


def test_batch_sync_filter_accumulates_like_the_sequential_one():
    rng = np.random.default_rng(1)
    seq, bat = SequentialFilter(5, clip=4.0), BatchSyncFilter(5, clip=4.0)
    for it in range(3):
        batch = rng.normal(1.0, 3.0, size=(64, 5))
        for row in batch:
            y = seq(row)
            assert np.all(np.abs(y) <= 4.0)
        bat(batch)
        bat.sync()
        np.testing.assert_allclose(bat.rs.M, seq.rs.M, rtol=1e-12)
        np.testing.assert_allclose(bat.rs.var, seq.rs.var, rtol=1e-12)
    y = bat(np.array([[1.0, 1.0, 1.0, 1.0, 100.0]]), update=False)
    assert y[0, 4] == 4.0 and abs(y[0, 0]) < 1.0


@pytest.mark.parametrize("demean,destd", [(True, True), (False, True), (True, False)])
def test_filters_subtract_the_mean_and_divide_by_the_std_only_when_asked(demean, destd):
    """RLlib's MeanStdFilter flags: subtract the mean only if demean, divide by std + 1e-8 only if destd, then clip.  The
    running statistics are kept either way."""
    rng = np.random.default_rng(2)
    seq = SequentialFilter(5, clip=4.0, demean=demean, destd=destd)
    bat = BatchSyncFilter(5, clip=4.0, demean=demean, destd=destd)
    for it in range(3):
        batch = rng.normal(1.0, 3.0, size=(64, 5))
        for row in batch:
            seq(row)
        bat(batch)
        bat.sync()
    np.testing.assert_allclose(bat.rs.M, seq.rs.M, rtol=1e-12)
    np.testing.assert_allclose(bat.rs.var, seq.rs.var, rtol=1e-12)
    assert bat.rs.n == seq.rs.n == 192
    probe = np.array([[1.0, 1.0, 1.0, 1.0, 100.0], [0.5, -2.0, 3.0, 0.25, -1.5]])
    want = probe - seq.rs.M if demean else probe.copy()
    if destd:
        want = want / (seq.rs.std + 1e-8)
    want = np.clip(want, -4.0, 4.0)
    assert want[0, 4] == 4.0                                   # clipped whatever the flags
    np.testing.assert_allclose(np.stack([seq(row, update=False) for row in probe]), want, rtol=1e-15, atol=0)
    np.testing.assert_allclose(bat(probe, update=False), want, rtol=0, atol=1e-6)      # float32 applied statistics
