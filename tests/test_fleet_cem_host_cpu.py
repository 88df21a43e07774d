"""Host-side argument checks of fleet.CemFleet that run before any device is touched."""
import pytest


def test_cem_fleet_rejects_before_creating_a_handle():
    from cartpolesimulation_b200.fleet import CemFleet
    with pytest.raises(NotImplementedError):
        CemFleet(4, integrator="neural")
    with pytest.raises(ValueError):
        CemFleet(4, noise="gaussian")
    with pytest.raises(ValueError):
        CemFleet(4, dt=0.02, dt_simulation=0.003)   # the plant period must be a whole number of ticks


def test_cem_fleet_config_struct_matches_header():
    import ctypes as C

    from cartpolesimulation_b200 import _lib as L
    # 4 ints, double, u64, i64, 3 ints, 2 floats -> 4*4 + 8 + 8 + 8 + 3*4 + 2*4 = 60, padded to the double's 8 -> 64
    assert C.sizeof(L.cps_cem_fleet_config) == 64
