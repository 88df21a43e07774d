"""Host-side argument checks of fleet.RandomActionFleet that run before any device is touched."""
import pytest


def test_random_action_fleet_rejects_before_creating_a_handle():
    from cartpolesimulation_b200.fleet import RandomActionFleet
    with pytest.raises(NotImplementedError):
        RandomActionFleet(4, integrator="neural")
    with pytest.raises(ValueError):
        RandomActionFleet(4, noise="gaussian")
    with pytest.raises(ValueError):
        RandomActionFleet(4, dt=0.02, dt_simulation=0.003)   # the plant period must be a whole number of ticks


def test_random_action_fleet_set_plant_models_is_not_offered():
    from cartpolesimulation_b200.fleet import RandomActionFleet
    with pytest.raises(NotImplementedError):
        RandomActionFleet.set_plant_models(object.__new__(RandomActionFleet), latency=0.01)


def test_random_action_fleet_config_struct_matches_header():
    import ctypes as C

    from cartpolesimulation_b200 import _lib as L
    # 4 ints, double, u64, i64 -> 4*4 + 8 + 8 + 8 = 40
    assert C.sizeof(L.cps_random_action_fleet_config) == 40
