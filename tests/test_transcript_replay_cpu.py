"""The product's host control flow consuming the CUDA solver's QP answers, with nothing from outside the repository.

tests/golden/cp20_transcript.npz freezes, on the golden noisy CP20 trajectory, every node QP kernel K1 answered, what
the device-side search K3 explored and what the device-side warm start K2+K4 produced; the unmodified reference
controller replayed through it reproduces it (tests/test_reference_replay_cpu.py, which needs the reference's sources).
Here the product's own restatement of that control flow -- ``feedforward`` / ``construct_warm_start`` with
``device_search = False``: one ``BoundedQP`` solve per node, the batched host warm start -- is replayed through the same
transcript, its device call answered from it.  Asserted, as for the reference:

* the host loop asks EXACTLY the QPs the device search solved, in the same order, with the same starts (bit for bit);
* explored node sequence, leaves (identifiers, order) and their lower bounds are bit-identical to K3; optimal cost too;
* the host warm start equals K2+K4: same cover, identifiers, order, dual = None pattern; bounds and dual objectives to
  1e-11 (the two sum the same terms in a different order); every root starts from its shifted multipliers.
"""
import numpy as np

from oracle.models import load_model
from tests.util import make_controller
from tests.test_reference_replay_cpu import TRANSCRIPT, _key, _idents


def test_host_control_flow_on_gpu_answers_equals_device_search():
    model = load_model('cp20')
    z = np.load(TRANSCRIPT)
    ctl = make_controller(model)
    ctl.device_search = False
    pd = ctl.problem
    table = {_key(z['qp_x0'][i], z['qp_lb'][i], z['qp_ub'][i], z['qp_y0'][i], z['qp_yc0'][i]): i
             for i in range(len(z['qp_status']))}
    asked = []

    def launch(x0, lb, ub, y0, yc0):
        k = _key(x0, lb, ub, np.zeros(pd.m) if y0 is None else y0, np.zeros(pd.n) if yc0 is None else yc0)
        assert k in table, 'the host loop asked a QP (or a start) the device search never solved'
        i = table[k]
        assert bool(z['qp_hot'][i]) == (y0 is not None)
        asked.append(i)
        return dict(status=z['qp_status'][i], cost=z['qp_cost'][i], dobj=z['qp_dobj'][i], iters=z['qp_iters'][i],
                    primal=z['qp_primal'][i], dual=z['qp_dual'][i], yc=z['qp_yc'][i], runtime=0.)
    ctl.qp._launch = launch
    nub = int(model['nub'])
    T, nx, nu = ctl.T, ctl.mld.nx, ctl.mld.nu
    ws = None
    x = model['x0_nominal'].copy()
    for t in range(int(z['n_steps'])):
        assert np.array_equal(x, z['k3_%d_x' % t])
        asked.clear()
        sol, leaves, n_qp, _ = ctl.feedforward(x, warm_start=ws, printing_period=None)
        c0, c1 = z['k3_%d_calls' % t]
        assert n_qp == c1 - c0
        assert asked == list(range(c0, c1))
        order = _idents(z['k3_%d_order_depth' % t], z['k3_%d_order_bits' % t], nub)
        for i, ident in zip(asked, order):
            lb, ub = ctl._get_bound_binaries(ident)
            assert np.array_equal(lb.ravel(), z['qp_lb'][i]) and np.array_equal(ub.ravel(), z['qp_ub'][i])
        dev = _idents(z['k3_%d_leaf_depth' % t], z['k3_%d_leaf_bits' % t], nub)
        assert [l.identifier for l in leaves] == dev
        assert np.array_equal(np.array([l.lb for l in leaves]), z['k3_%d_leaf_lb' % t])
        assert sol.objective == float(z['k3_%d_cost' % t])
        U = z['k3_%d_primal' % t][(T + 1) * nx:].reshape(T, nu)
        assert np.array_equal(np.array(sol.variables['ub']), U[:, nu - nub:])
        e = z['k4_%d_e' % t]
        ws, _, _ = ctl.construct_warm_start(leaves, x, sol.variables['uc'][0], sol.variables['ub'][0], e)
        assert [l.identifier for l in ws] == _idents(z['k4_%d_depth' % t], z['k4_%d_bits' % t], nub)
        lb_host, lb_dev = np.array([l.lb for l in ws]), z['k4_%d_lb' % t]
        assert np.array_equal(np.isinf(lb_host), np.isinf(lb_dev))
        fin = np.isfinite(lb_dev)
        scale = max(1., np.abs(z['k4_%d_dobj' % t]).max())
        assert np.all(np.abs(lb_host[fin] - lb_dev[fin]) <= 1e-11 * scale)
        none = np.array([l.extra.dual is None for l in ws])
        assert np.array_equal(none, z['k4_%d_none' % t])
        dobj = np.array([0. if l.extra.dual is None else l.extra.dual.objective for l in ws])
        assert np.all(np.abs(dobj[~none] - z['k4_%d_dobj' % t][~none]) <= 1e-11 * scale)
        # the roots' starts are the device's to rounding; take the device's bits so that the next step's requests can be
        # looked up in the transcript
        for j, l in enumerate(ws):
            a = dict(c=list(z['k4_%d_start_c' % t][j]), v=list(z['k4_%d_start_v' % t][j]))
            if l.extra.dual is not None:
                assert np.allclose(l.extra.active_set['c'], a['c'], rtol=1e-12, atol=1e-13)
            l.extra.active_set = a
        x = sol.variables['x'][1] + e
