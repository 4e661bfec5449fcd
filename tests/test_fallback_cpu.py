"""The host side of the fallback policy (wshmpc_fallback): the struct's packing against the C header, the argument checks of
ClosedLoop(..., fallback=H) that need no GPU, and a numpy statement of the policy table that the GPU tests replay."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def policy(live, has_inc, status, age, H):
    """The policy of one instance-step (include/wshmpc.h, wshmpc_fallback), elementwise on numpy arrays:
    returns (source, hold, active after the step, age after the step); source 0 the incumbent, 1 the plan, -1 none."""
    live, has_inc = np.asarray(live, bool), np.asarray(has_inc, bool)
    status, age = np.asarray(status), np.asarray(age)
    inc = live & has_inc
    plan = live & ~has_inc & (status == 1) & (age >= 0) & (age + 1 <= H)
    source = np.where(inc, 0, np.where(plan, 1, -1))
    hold = np.where(inc, 0, np.where(plan, age + 1, -1))
    new_age = np.where(inc, 0, np.where(plan, age + 1, age))
    return source, hold, (source >= 0).astype(int), new_age


def replay(status, cost, H, active0=None):
    """hold [n_steps, n_inst] the policy gives to the logs of a loop (status, cost [n_steps, n_inst]) started without plans"""
    S, N = status.shape
    live = np.ones(N, bool) if active0 is None else np.asarray(active0, bool)
    age = np.full(N, -1)
    hold = np.zeros((S, N), dtype=int)
    for t in range(S):
        _, hold[t], act, age = policy(live, np.isfinite(cost[t]), status[t], age, H)
        live = act.astype(bool)
    return hold


def test_policy_table_hand_built_cases():
    H = 3
    # (live, has incumbent, status, age) -> (source, hold, active, age after)
    cases = [
        ((1, 1, 0, -1), (0, 0, 1, 0)),     # first incumbent: a plan from now on
        ((1, 1, 0, 2), (0, 0, 1, 0)),      # an incumbent renews the plan
        ((1, 1, 2, 1), (0, 0, 1, 0)),      # capacity with an incumbent: applied as today
        ((1, 0, 1, -1), (-1, -1, 0, -1)),  # infeasible without a plan: off
        ((1, 0, 1, 0), (1, 1, 1, 1)),      # infeasible, plan of age 0: u_1
        ((1, 0, 1, 2), (1, 3, 1, 3)),      # ... age 2: u_3 = the last step H allows
        ((1, 0, 1, 3), (-1, -1, 0, 3)),    # plan used up: off
        ((1, 0, 2, 0), (-1, -1, 0, 0)),    # capacity without an incumbent: no complete cover to shift, off
        ((1, 0, 3, 0), (-1, -1, 0, 0)),    # QP iteration limit: off
        ((0, 0, 1, 0), (-1, -1, 0, 0)),    # an instance already off stays off
        ((0, 1, 0, 0), (-1, -1, 0, 0)),
    ]
    for (lv, hi, st, a), want in cases:
        got = tuple(int(np.asarray(v)) for v in policy(lv, hi, st, a, H))
        assert got == want, ((lv, hi, st, a), got, want)
    # H = 0 is the loop without a fallback: an instance stays exactly while it has incumbents
    for st in (0, 1, 2, 3):
        for a in (-1, 0, 5):
            for hi in (0, 1):
                src, hold, act, _ = policy(1, hi, st, a, 0)
                assert int(act) == hi and int(hold) == (0 if hi else -1)


def test_replay_runs_of_holds():
    inf = np.inf
    # one instance: solved, 3 infeasible steps, solved, 4 infeasible steps (the plan runs out after H = 3)
    status = np.array([0, 1, 1, 1, 0, 1, 1, 1, 1, 1])[:, None]
    cost = np.where(status == 0, 1., inf)
    assert replay(status, cost, 3)[:, 0].tolist() == [0, 1, 2, 3, 0, 1, 2, 3, -1, -1]
    assert replay(status, cost, 1)[:, 0].tolist() == [0, 1, -1, -1, -1, -1, -1, -1, -1, -1]
    assert replay(status, cost, 0)[:, 0].tolist() == [0] + [-1] * 9
    # infeasible at step 0: no plan yet
    assert replay(np.array([[1], [0]]), np.array([[inf], [1.]]), 19)[:, 0].tolist() == [-1, -1]


def test_fallback_struct_packing():
    import ctypes as C
    import torch
    from warm_start_hmpc_b200 import capi
    N, P = 5, 224
    fb = dict(max_hold=3, plan=torch.zeros((N, P), dtype=torch.float64), age=torch.full((N,), -1, dtype=torch.int32),
              app_cost=torch.zeros(N, dtype=torch.float64), app_primal=torch.zeros((N, P), dtype=torch.float64))
    hold = torch.zeros((7, N), dtype=torch.int32)
    c = capi._fallback_struct(fb, hold)
    assert c.max_hold == 3 and c.d_plan == fb['plan'].data_ptr() and c.d_age == fb['age'].data_ptr()
    assert c.d_app_cost == fb['app_cost'].data_ptr() and c.d_app_primal == fb['app_primal'].data_ptr()
    assert c.d_hold == hold.data_ptr()
    assert capi._fallback_struct(dict(fb, plan=None), None).d_plan is None
    assert 'wshmpc_closed_loop_fallback' in capi.EXPORTS and 'wshmpc_fallback_step' in capi.EXPORTS
    # the ctypes layout is the C layout of include/wshmpc.h
    fields = [f for f, _ in capi._Fallback._fields_]
    src = '#include <stddef.h>\n#include <stdio.h>\n#include "wshmpc.h"\nint main(void) {\n'
    src += ''.join('printf("%%zu\\n", offsetof(wshmpc_fallback, %s));\n' % f for f in fields)
    src += 'printf("%zu\\n", sizeof(wshmpc_fallback)); return 0; }\n'
    with tempfile.TemporaryDirectory() as d:
        with open(os.path.join(d, 'm.c'), 'w') as f:
            f.write(src)
        subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), '-o', os.path.join(d, 'm'), os.path.join(d, 'm.c')])
        out = [int(v) for v in subprocess.check_output([os.path.join(d, 'm')]).split()]
    assert out[:-1] == [getattr(capi._Fallback, f).offset for f in fields]
    assert out[-1] == C.sizeof(capi._Fallback)


@pytest.fixture(scope='module')
def ctl():
    from oracle.models import load_model
    from tests.util import make_controller
    return make_controller(load_model('cp20'))


@pytest.mark.parametrize('H', [-1, 20, 25, 1.5])
def test_max_hold_range(ctl, H):
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    assert ctl.T == 20
    with pytest.raises(ValueError, match='fallback'):
        ClosedLoop(ctl, 4, fallback=H)


def test_closed_loop_value_errors(ctl):
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    with pytest.raises(ValueError, match='comparator'):
        ClosedLoop(ctl, 4, warm=False, comparator=True, fallback=3)
    # run_mailbox and rebalance refuse a loop with plans before they touch the device
    L = ClosedLoop.__new__(ClosedLoop)
    L.plant, L.fb = None, dict(max_hold=3)
    with pytest.raises(ValueError, match='fallback'):
        L.run_mailbox(1, lambda *a: None)
    with pytest.raises(ValueError, match='fallback plans'):
        L.rebalance()
