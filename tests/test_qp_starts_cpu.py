"""CPU: the start generators of tests/test_gpu_qp_starts.py produce what they claim, and the CPU stand-in of the device
call (tests/util.oracle_launch) ignores the start entries K1 ignores."""
import numpy as np
import pytest

from oracle.models import load_model
from tests.util import (make_problem, random_nodes, prefix_depth, record_to_y0, y0_to_multipliers, sparse_start,
                        dense_start, wide_start, out_of_contract, start_rows, oracle_launch)


@pytest.fixture(scope='module')
def cp20():
    model = load_model('cp20')
    return model, make_problem(model)


def _stage(pd, r):
    """Time step of row r: stage rows come in blocks of nh (the last block holds nh1), bound rows in blocks of nub."""
    return min(r // pd.nh, pd.T - 1) if r < pd.mc else (r - pd.mc) // pd.nub


@pytest.mark.parametrize('d', [0, 3, 8])
def test_wide_starts_have_the_claimed_rank_spread_over_all_stages(cp20, d):
    model, pd = cp20
    y, rank = wide_start(np.random.default_rng(d), pd, d, 100)
    rows = np.nonzero(y)[0]
    assert rows.size <= pd.n                                  # no truncation to n rows
    assert rank >= 100 and np.linalg.matrix_rank(pd.Mh[rows][:, d:]) == rank
    assert not np.any((rows >= pd.mc) & (rows < pd.mc + d))   # no row the node eliminates
    assert {_stage(pd, r) for r in rows} == set(range(pd.T))
    assert np.all(y[rows[rows < pd.mc]] > 0.)
    assert np.all(start_rows(y, pd.mc) == (y != 0.))         # every entry enters


def test_sparse_and_dense_starts(cp20):
    model, pd = cp20
    rng = np.random.default_rng(0)
    for k in (1, 7, 20):
        y = sparse_start(rng, pd, k)
        assert np.count_nonzero(y) == k and np.all(y[:pd.mc] >= 0.)
        a = np.abs(y[y != 0.])
        assert a.min() >= 1e-8 and a.max() <= 1e8
    y = dense_start(rng, pd)
    assert np.all(y != 0.) and np.all(y[:pd.mc] > 0.) and np.any(y[pd.mc:] < 0.)


def test_record_y0_round_trip(cp20):
    """[mu | nu_ub - nu_lb] and back: the multipliers of a record (at most one side of a binary non-zero, as K1 writes
    them) are recovered exactly; the other families do not enter."""
    model, pd = cp20
    L = pd.layout
    rng = np.random.default_rng(1)
    dual = rng.standard_normal((3, L.dual))
    y = rng.standard_normal((3, pd.m))
    dual[:, L.off_mu:L.off_nu_lb] = np.maximum(y[:, :pd.mc], 0.)
    dual[:, L.off_nu_lb:L.off_nu_ub] = np.maximum(-y[:, pd.mc:], 0.)
    dual[:, L.off_nu_ub:L.off_rho] = np.maximum(y[:, pd.mc:], 0.)
    y0 = record_to_y0(dual, L)
    assert y0.shape == (3, pd.m)
    mu, nl, nu = y0_to_multipliers(y0, pd.mc)
    assert np.array_equal(mu, dual[:, L.off_mu:L.off_nu_lb])
    assert np.array_equal(nl, dual[:, L.off_nu_lb:L.off_nu_ub]) and np.array_equal(nu, dual[:, L.off_nu_ub:L.off_rho])
    assert np.array_equal(y0[:, pd.mc:], np.where(y[:, pd.mc:] > 0., y[:, pd.mc:], np.where(y[:, pd.mc:] < 0., y[:, pd.mc:], 0.)))


def test_deeper_prefix_rows_are_the_eliminated_ones(cp20):
    """A start taken from a node with a deeper pinned prefix carries multipliers on bound rows mc + j, j < d, of the
    node it starts: rows that node eliminates (K1 skips them)."""
    model, pd = cp20
    x0, lb, ub = random_nodes(model, 8, seed=3)
    deep, shallow = 0, 1
    lb[deep, :40] = ub[deep, :40] = 0.; lb[shallow] = 0.; ub[shallow] = 1.; lb[shallow, :5] = ub[shallow, :5] = 0.
    assert prefix_depth(lb[deep], ub[deep], pd.n_elim) == 40 and prefix_depth(lb[shallow], ub[shallow], pd.n_elim) == 5
    launch = oracle_launch(model, pd)
    out = launch(x0[deep], lb[deep], ub[deep], None, None)
    y0 = record_to_y0(out['dual'], pd.layout)
    assert np.count_nonzero(y0[pd.mc:pd.mc + 5]) > 0


def test_prefix_depth_stops_at_the_first_free_binary_and_at_n_elim():
    lb, ub = np.zeros(10), np.ones(10)
    assert prefix_depth(lb, ub, 10) == 0
    lb[:4] = ub[:4] = 1.; lb[6] = ub[6] = 0.
    assert prefix_depth(lb, ub, 10) == 4 and prefix_depth(lb, ub, 3) == 3
    assert prefix_depth(np.ones(10), np.ones(10), 10) == 10


def test_out_of_contract_entries_are_what_a_start_ignores(cp20):
    model, pd = cp20
    rng = np.random.default_rng(2)
    y = sparse_start(rng, pd, 12)
    bad = out_of_contract(rng, y, pd.mc)
    assert np.isnan(bad).sum() == 3 and np.isposinf(bad).sum() == 3 and np.isneginf(bad).sum() == 3
    assert np.sum((bad < 0.) & np.isfinite(bad) & (np.arange(pd.m) < pd.mc)) == 3
    assert np.array_equal(start_rows(bad, pd.mc), start_rows(y, pd.mc))
    assert np.array_equal(np.where(start_rows(bad, pd.mc), bad, 0.), y)


def test_oracle_launch_ignores_out_of_contract_entries(cp20):
    """The CPU replay of the device call applies the same rule as K1: the solve from a start with negative stage-row
    entries, NaN and +-inf is the solve from the start without them."""
    model, pd = cp20
    launch = oracle_launch(model, pd)
    x0, lb, ub = random_nodes(model, 4, seed=6)
    rng = np.random.default_rng(4)
    for i in range(4):
        y = sparse_start(rng, pd, 10)
        a = launch(x0[i], lb[i], ub[i], y, None)
        b = launch(x0[i], lb[i], ub[i], out_of_contract(rng, y, pd.mc), None)
        assert a['status'] == b['status'] and a['iters'] == b['iters']
        assert np.array_equal(a['dual'], b['dual']) and np.array_equal(a['primal'], b['primal'])
