"""Host-side checks of fleet.Fleet's `network` keyword that run before any device is touched."""
import pytest


def test_neural_fleet_needs_its_network():
    from cartpolesimulation_b200.fleet import Fleet
    with pytest.raises(NotImplementedError, match="network="):
        Fleet(4, 64, 10, integrator="neural")
    with pytest.raises(NotImplementedError, match="network="):
        Fleet(4, 64, 10, integrator="neural", net_kernel="fp32")


def test_network_belongs_to_the_neural_predictor_only():
    from cartpolesimulation_b200.fleet import Fleet
    spec = dict(net_type="GRU", hsz=[32, 32])
    for integrator in ("ODE", "ODE_v0"):
        with pytest.raises(ValueError, match="network"):
            Fleet(4, 64, 10, integrator=integrator, network=spec)
