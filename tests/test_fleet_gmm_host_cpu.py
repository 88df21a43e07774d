"""Host-side argument checks of fleet.CemGmmFleet that run before any device is touched."""
import pytest


def test_cem_gmm_fleet_rejects_before_creating_a_handle():
    from cartpolesimulation_b200.fleet import CemGmmFleet
    with pytest.raises(NotImplementedError):
        CemGmmFleet(4, integrator="neural")
    with pytest.raises(ValueError):
        CemGmmFleet(4, noise="gaussian")
    with pytest.raises(ValueError):
        CemGmmFleet(4, dt=0.02, dt_simulation=0.003)   # the plant period must be a whole number of ticks


def test_cem_gmm_fleet_set_plant_models_is_not_offered():
    from cartpolesimulation_b200.fleet import CemGmmFleet
    with pytest.raises(NotImplementedError):
        CemGmmFleet.set_plant_models(object.__new__(CemGmmFleet), latency=0.01)


def test_cem_gmm_fleet_config_struct_matches_header():
    import ctypes as C

    from cartpolesimulation_b200 import _lib as L
    # 4 ints, double, u64, i64, 2 ints, 2 floats -> 4*4 + 8 + 8 + 8 + 2*4 + 2*4 = 56
    assert C.sizeof(L.cps_cem_gmm_fleet_config) == 56
