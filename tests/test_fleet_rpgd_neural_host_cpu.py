"""Host-side checks of fleet.RpgdFleet's `network` keyword that run before any device is touched."""
import pytest


def test_neural_rpgd_fleet_needs_its_network():
    from cartpolesimulation_b200.fleet import RpgdFleet
    with pytest.raises(NotImplementedError, match="network="):
        RpgdFleet(4, integrator="neural")


def test_network_belongs_to_the_neural_predictor_only():
    from cartpolesimulation_b200.fleet import RpgdFleet
    spec = dict(net_type="GRU", hsz=[32, 32])
    for integrator in ("ODE", "ODE_v0"):
        with pytest.raises(ValueError, match="network"):
            RpgdFleet(4, integrator=integrator, network=spec)
