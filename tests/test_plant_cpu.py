"""The host side of the device plant (plants.DevicePlant): parameter packing, the Euler sub-step rule of
CartPoleWithWalls.simulate, and the argument checks that need no GPU."""
import numpy as np
import pytest


def test_params_packing():
    from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant
    p = CartPoleWithWalls(mc=1.1, mp=.9, l=1.2, d=.45, stiffness=120., damping=8., g=9.81)
    assert np.array_equal(p.params(), [1.1, .9, 1.2, .45, 120., 8., 9.81])
    assert np.array_equal(CartPoleWithWalls().params(), [1., 1., 1., .5, 100., 10., 10.])
    one = DevicePlant(p, .05, device='cpu')
    assert one.n_sets == 1 and str(one.params.dtype) == 'torch.float64' and one.n_sub == 50
    assert np.array_equal(one.params.numpy(), p.params()[None])
    ps = [CartPoleWithWalls(mp=.7 + .1 * k) for k in range(5)]
    many = DevicePlant(ps, .05, fc_index=2, device='cpu')
    assert many.n_sets == 5 and many.fc_index == 2 and many.params.is_contiguous()
    assert np.array_equal(many.params.numpy(), np.stack([q.params() for q in ps]))


@pytest.mark.parametrize('dt, h_des, n', [(.05, 1e-3, 50), (.05, 2e-3, 25), (1e-4, 1e-3, 1), (.0525, 1e-3, 52), (.1, .03, 3)])
def test_n_sub_follows_simulate(dt, h_des, n):
    from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant, n_substeps
    assert n_substeps(dt, h_des) == n
    assert DevicePlant(CartPoleWithWalls(), dt, h_des, device='cpu').n_sub == n
    # simulate takes the same number of sub-steps: n explicit Euler steps of dt / n by hand
    p, x, fc = CartPoleWithWalls(), np.array([.3, .1, -.4, .2]), .5
    y = x.copy()
    for _ in range(n):
        y = y + dt / n * p.x_dot(y, np.asarray(fc))
    assert np.array_equal(p.simulate(x, dt, fc, h_des), y)


def test_device_plant_argument_errors():
    from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant
    p = CartPoleWithWalls()
    with pytest.raises(ValueError, match='CartPoleWithWalls'):
        DevicePlant([], .05, device='cpu')
    with pytest.raises(ValueError, match='CartPoleWithWalls'):
        DevicePlant([p, object()], .05, device='cpu')
    with pytest.raises(ValueError, match='dt'):
        DevicePlant(p, 0., device='cpu')
    with pytest.raises(ValueError, match='dt'):
        DevicePlant(p, .05, h_des=-1e-3, device='cpu')
    with pytest.raises(ValueError, match='fc_index'):
        DevicePlant(p, .05, fc_index=-1, device='cpu')
    with pytest.raises(ValueError, match='fc_index'):
        DevicePlant(p, .05, fc_index=.5, device='cpu')
