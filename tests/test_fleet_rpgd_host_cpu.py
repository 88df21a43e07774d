"""Host-side argument checks of fleet.RpgdFleet that run before any device is touched."""
import pytest


def test_rpgd_fleet_rejects_before_creating_a_handle():
    from cartpolesimulation_b200.fleet import RpgdFleet
    with pytest.raises(NotImplementedError):
        RpgdFleet(4, SAMPLING_DISTRIBUTION="uniform")
    with pytest.raises(ValueError):
        RpgdFleet(4, SAMPLING_DISTRIBUTION="beta")
    with pytest.raises(ValueError):
        RpgdFleet(4, noise="gaussian")
    with pytest.raises(ValueError):
        RpgdFleet(4, dt=0.02, dt_simulation=0.003)   # the plant period must be a whole number of ticks


def test_rpgd_fleet_config_struct_matches_header():
    import ctypes as C

    from cartpolesimulation_b200 import _lib as L
    # 4 ints, double, u64, i64, 5 ints, 7 floats -> 4*4 + 8 + 8 + 8 + 5*4 + 7*4 = 88
    assert C.sizeof(L.cps_rpgd_fleet_config) == 88
