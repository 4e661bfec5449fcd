"""The host side of the closed loop's per-step statistics (wshmpc_loop d_log_cover, d_log_lapsed, d_log_iters;
ClosedLoop(..., stats=True)): the struct's packing against the C header, the argument check that needs no GPU, and the
oracle's cover and lapsed counts on the golden noisy trajectory, which tests/test_gpu_loop_stats.py holds the fused loop to."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# oracle/bnb_ref.py on the golden noisy CP20 trajectory (tests/golden/cp20_closed_loop.npz noisy_*, sigma = .003): per step,
# the roots of the warm start construct_warm_start hands to the next step, and how many of them have dual = None.  The device
# logs the same cover and, for steps 0-2, the same lapsed counts; from step 3 on its search ends with Farkas proofs that survive
# the shift where some of the oracle's lapse (DESIGN section 5), and its lapsed counts are checked against the oracle's
# construct_warm_start on the device's own leaves instead.
GOLDEN_NOISY_COVER = [77, 77, 77, 77, 77, 77]
GOLDEN_NOISY_LAPSED = [2, 3, 1, 3, 2, 1]


def test_loop_struct_packing():
    import ctypes as C
    from warm_start_hmpc_b200 import capi
    fields = [f for f, _ in capi._Loop._fields_]
    assert fields[-3:] == ['d_log_cover', 'd_log_lapsed', 'd_log_iters']
    src = '#include <stddef.h>\n#include <stdio.h>\n#include "wshmpc.h"\nint main(void) {\n'
    src += ''.join('printf("%%zu\\n", offsetof(wshmpc_loop, %s));\n' % f for f in fields)
    src += 'printf("%zu\\n", sizeof(wshmpc_loop)); return 0; }\n'
    with tempfile.TemporaryDirectory() as d:
        with open(os.path.join(d, 'm.c'), 'w') as f:
            f.write(src)
        subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), '-o', os.path.join(d, 'm'), os.path.join(d, 'm.c')])
        out = [int(v) for v in subprocess.check_output([os.path.join(d, 'm')]).split()]
    assert out[:-1] == [getattr(capi._Loop, f).offset for f in fields]
    assert out[-1] == C.sizeof(capi._Loop)
    # a zero-initialised struct asks for none of the statistics
    L = capi._Loop()
    assert L.d_log_cover is None and L.d_log_lapsed is None and L.d_log_iters is None


@pytest.mark.parametrize('stats', [1, 0, 'yes', None, 2.])
def test_stats_argument(stats):
    """stats is True or False; anything else fails before the device is touched"""
    from oracle.models import load_model
    from tests.util import make_controller
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    ctl = make_controller(load_model('cp20'))
    with pytest.raises(ValueError, match='stats'):
        ClosedLoop(ctl, 4, stats=stats)


def test_oracle_cover_and_lapsed_on_the_golden_noisy_trajectory():
    """construct_warm_start of oracle/bnb_ref.py along the reference's noisy trajectory: the published cover of 77 every
    step, and the lapsed (dual = None) counts the GPU tests hold the fused loop to"""
    from oracle.models import load_model, GOLDEN
    from oracle.qp_c import CoreC
    from oracle.bnb_ref import OracleController
    model = load_model('cp20')
    g = np.load(os.path.join(GOLDEN, 'cp20_closed_loop.npz'))
    ctl = OracleController(model, CoreC(model, variant=1), hot_start='record')
    x = np.array(model['x0_nominal'], dtype=float)
    ws = None
    cover, lapsed = [], []
    for t, e in enumerate(g['noisy_e']):
        assert np.allclose(x, g['noisy_x'][t], rtol=0, atol=1e-7), t
        inc, leaves, _ = ctl.feedforward(x, warm_start=ws)
        u0 = inc.primal['u'][0]
        ws = ctl.construct_warm_start(leaves, x, u0[:ctl.nuc], u0[ctl.nuc:], e)
        cover.append(len(ws))
        lapsed.append(sum(n.dual is None for n in ws))
        x = inc.primal['x'][1] + e
    assert cover == GOLDEN_NOISY_COVER == [int(c) for c in g['noisy_cover']]
    assert lapsed == GOLDEN_NOISY_LAPSED
