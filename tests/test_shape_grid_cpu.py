"""The shape grid (tests/shape_grid.py) without a GPU: it reaches every branch condition it is there for, the record
layout the CPU code computes is the library's, the oracle answers are certified before the kernels are judged by them,
and the elimination overrides are valid inputs."""
import numpy as np
import pytest

from oracle.condense import Condensed
from oracle.models import load_model
from tests import shape_grid as sg
from tests.util import check_node_result, make_problem, oracle_launch


def test_grid_reaches_every_listed_condition():
    reached = {}
    for s in sg.GRID:
        for c in sg.conditions(s):
            reached.setdefault(c, []).append(s.name)
    missing = [c for c in sg.COVERAGE if c not in reached]
    assert not missing, 'no shape of the grid reaches: %s' % ', '.join(missing)
    assert 'n_elim out of range' not in reached


def test_conditions_name_what_an_edited_grid_loses():
    """The coverage check fails, and names the condition, when the only shape that reaches it leaves the grid."""
    for name, cond in (('n513', 'n > 512 refused'), ('nx33', 'nx > 32'), ('odd_rec', 'shift stages records that dual + n would misalign'),
                       ('nub32', 'H = T - 1 == 1')):
        rest = [s for s in sg.GRID if s.name != name]
        reached = set().union(*(sg.conditions(s) for s in rest))
        assert cond not in reached, (name, cond)


@pytest.mark.parametrize('name', ['cp20', 'cp40', 'cp1w40', 'syn30'])
def test_record_stride_of_the_shipped_models_is_unchanged(name):
    L = sg.dims(load_model(name))['layout']
    n = sg.dims(load_model(name))['n']
    assert L.rec_stride == L.dual + n and L.rec_stride % 2 == 0


@pytest.mark.parametrize('shape', sg.GRID, ids=str)
def test_record_stride_is_even_and_holds_the_record(shape):
    d = sg.dims(shape.model())
    L = d['layout']
    assert L.rec_stride % 2 == 0 and L.dual + d['n'] <= L.rec_stride <= L.dual + d['n'] + 1
    # the generator is deterministic: the same call gives the same bits
    m2 = sg._model.__wrapped__(shape.name)
    assert all(np.array_equal(np.asarray(shape.model()[k]), np.asarray(m2[k])) for k in ('A', 'B', 'F', 'G', 'h', 'x0_nominal'))


def test_issue_dimensions_of_the_misaligned_shape():
    """odd_rec is the example of the defect: n = 35, dual = 258, so dual + n = 293 is odd and the stride is 294."""
    d = sg.dims(sg.BY_NAME['odd_rec'].model())
    assert (d['n'], d['layout'].dual, d['layout'].rec_stride) == (35, 258, 294)
    assert sg.staging(d) == 'all'


ORACLE_SHAPES = [s for s in sg.GRID if s.tier in (sg.K3, sg.ALL)]


@pytest.mark.parametrize('shape', ORACLE_SHAPES, ids=str)
def test_oracle_answers_are_certified(shape):
    """20 nodes per shape through the oracle's QP core (the thin factor of the CUDA kernel), each passed through the
    solver-independent certificates the GPU results are checked with."""
    model = shape.model()
    pd = make_problem(model)
    assert pd.layout.rec_stride == sg.dims(model)['layout'].rec_stride and pd.n_elim == pd.nb
    cond = Condensed(model)
    launch = oracle_launch(model, pd)
    x0, lb, ub = sg.nodes(shape, 20, seed=1, opt=sg.oracle_optimum(shape))
    seen = set()
    for i in range(len(x0)):
        r = launch(x0[i], lb[i], ub[i], None, None)
        seen.add(r['status'])
        check_node_result(model, cond, pd, pd.layout, x0[i], lb[i], ub[i], r['status'], r['cost'], r['dobj'], r['primal'],
                          r['dual'], tag=(shape.name, i))
    assert seen == {2, 3}, (shape.name, seen)                # optimal and infeasible nodes both


ELIM_SHAPES = [s for s in sg.GRID if s.elim]


@pytest.mark.parametrize('shape', ELIM_SHAPES, ids=str)
def test_elimination_overrides_are_valid_inputs(shape):
    """For n_elim = k, Linv[:k, :k] is the inverse of the leading k x k block of the binaries' bound rows Mh[mc:, :nb] (lower
    triangular, so the leading block of its inverse is the inverse of its leading block), and 0 <= k <= nb."""
    pd0 = make_problem(shape.model())
    L = pd0.Mh[pd0.mc:, :pd0.nb]
    assert np.allclose(L, np.tril(L), rtol=0, atol=0)
    for k in shape.elim:
        pd = sg.problem(shape, k)
        assert pd.n_elim == k and 0 <= k < pd.nb
        if k:
            prod = pd.Linv[:k, :k].dot(pd.Mh[pd.mc:pd.mc + k, :k])
            assert np.allclose(prod, np.eye(k), rtol=0, atol=1e-9), (shape.name, k, np.abs(prod - np.eye(k)).max())
