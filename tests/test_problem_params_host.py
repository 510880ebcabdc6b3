"""Per-problem parameters on the host: the record layout of cudampc_params as a NumPy dtype, params_array, and the checks
solve_batch / track_batch / start_batch run before any launch."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

from conftest import product_params


def test_params_dtype_is_the_c_record():
    from rrt_mpc_b200 import _lib
    assert _lib.PARAMS_DTYPE.itemsize == C.sizeof(_lib.Params) == 416
    assert list(_lib.PARAMS_DTYPE.names) == [f[0] for f in _lib.Params._fields_]
    for name, _ in _lib.Params._fields_:
        assert _lib.PARAMS_DTYPE.fields[name][1] == getattr(_lib.Params, name).offset, name
        assert _lib.PARAMS_DTYPE.fields[name][0].itemsize == getattr(_lib.Params, name).size, name


def test_params_array_round_trips_params_to_c():
    from rrt_mpc_b200 import params_array
    from rrt_mpc_b200.mpc_controller import params_to_c
    rng = np.random.default_rng(0)
    ps = []
    for k in range(5):
        q = rng.normal(size=(4, 4))
        ps.append(dataclasses.replace(product_params(20), wheelbase_px=3.0 + k, q=q @ q.T, du_bounds=((-k, k), (-0.1 * k, 0.2)),
                                      slack_rate=100.0 + k))
    arr = params_array(ps)
    assert arr.shape == (5,)
    for k, p in enumerate(ps):
        assert arr[k].tobytes() == bytes(params_to_c(p))
    assert arr["wheelbase_px"].tolist() == [3.0, 4.0, 5.0, 6.0, 7.0]
    assert arr["du_bounds"][3].tolist() == [-3.0, 3.0, -0.30000000000000004, 0.2]
    arr["du_bounds"][:, 3] = 0.05                                    # vectorised edits of a sweep
    assert (arr["du_bounds"][:, 3] == 0.05).all() and arr["du_bounds"][2, 2] == -0.2


def test_mismatched_params_raise_before_any_launch():
    from rrt_mpc_b200 import MPCConfig, MPCController, TrajectoryTracker, params_array
    base = product_params(20)
    ctl = MPCController(base, max_batch=4)
    x0, ref, up = np.zeros((3, 4)), np.zeros((3, 21, 4)), np.zeros((3, 2))
    cases = [
        ([base] * 2, "records"),                                               # wrong count
        ([base, base, dataclasses.replace(base, horizon=21)], "horizon"),
        ([base, dataclasses.replace(base, dt=base.dt * (1 + 2 ** -52)), base], "dt"),
        (params_array([base] * 3)[None], "records"),                          # wrong shape
        (np.zeros(3), "dtype"),
    ]
    for params, what in cases:
        with pytest.raises(ValueError, match=what):
            ctl.solve_batch(x0, ref, u_prev=up, params=params)
    assert ctl._h is None                                                     # no handle was created, nothing launched
    tr = TrajectoryTracker(MPCConfig(horizon=20), None)
    paths = [[(0.0, 0.0), (50.0, 0.0)]] * 2
    for call in (tr.track_batch, tr.start_batch):
        with pytest.raises(ValueError, match="horizon"):
            call(paths, np.zeros((2, 2)), np.ones((2, 2)), map_resolution=0.8,
                 vehicle_params=[MPCConfig(horizon=21).to_parameters(0.8)] * 2)
        with pytest.raises(ValueError, match="records"):
            call(paths, np.zeros((2, 2)), np.ones((2, 2)), map_resolution=0.8, vehicle_params=[MPCConfig(horizon=20).to_parameters(0.8)])
