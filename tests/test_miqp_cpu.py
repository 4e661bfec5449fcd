"""CPU: argument checks of the MIQP comparator's closed loop that come before any device work."""
import pytest

from oracle.models import load_model
from tests.util import make_controller


def test_comparator_rejects_warm_trees_before_touching_the_device():
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    ctl = make_controller(load_model('cp20'))
    with pytest.raises(ValueError, match='cold trees only'):
        ClosedLoop(ctl, 4, warm=True, comparator=True)
    assert ctl._handle is None                          # no handle was created


def test_device_comparator_runs_the_host_loop_for_other_methods():
    """feedforward_miqp_device starts children from their parent's record (Method = 1).  Any other Method solves every node
    from the empty working set, which only the host loop does: the call returns what feedforward_miqp returns.  (Device call
    of the QP seam replaced by the CPU oracle core: no GPU here.)"""
    import os
    import numpy as np
    from oracle.models import GOLDEN
    from tests.util import oracle_launch
    model = load_model('cp20')
    ctl = make_controller(model)
    ctl.qp._launch = oracle_launch(model, ctl.problem)
    x0 = np.load(os.path.join(GOLDEN, 'cp20_nodes.npz'))['x0']
    var_h, obj_h, nodes_h, _ = ctl.feedforward_miqp(x0, {'Method': 0})
    var_d, obj_d, nodes_d, _ = ctl.feedforward_miqp_device(x0, {'Method': 0})
    assert ctl._handle is None                          # no device search was started
    assert nodes_d == nodes_h and obj_d == obj_h
    for k in ('x', 'uc', 'ub'):
        assert np.array_equal(var_d[k], var_h[k])
