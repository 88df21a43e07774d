"""Host-side argument checks of fleet.LegacyFleet that run before any device is touched."""
import pytest


def test_legacy_fleet_rejects_before_creating_a_handle():
    from cartpolesimulation_b200.fleet import LegacyFleet
    with pytest.raises(NotImplementedError):
        LegacyFleet(4, predictor_specification="neural")
    with pytest.raises(NotImplementedError):
        LegacyFleet(4, cost_noise=0.1)           # would need cost weights per experiment
    with pytest.raises(ValueError):
        LegacyFleet(4, SAMPLING_TYPE="gaussian")
    with pytest.raises(ValueError):
        LegacyFleet(4, noise="gaussian")
    with pytest.raises(ValueError):
        LegacyFleet(4, dt=0.02, dt_simulation=0.003)   # the plant period must be a whole number of ticks


def test_legacy_fleet_set_plant_models_is_not_offered():
    from cartpolesimulation_b200.fleet import LegacyFleet
    with pytest.raises(NotImplementedError):
        LegacyFleet.set_plant_models(object.__new__(LegacyFleet), latency=0.01)


def test_legacy_fleet_config_struct_matches_header():
    import ctypes as C
    from cartpolesimulation_b200 import _lib as L
    # int x4, double, u64, i64, int sampling_type, int update_every, double stdev, double p_Q
    assert C.sizeof(L.cps_legacy_fleet_config) == 64
    assert L.cps_legacy_fleet_config.stdev.offset == 48 and L.cps_legacy_fleet_config.p_Q.offset == 56
