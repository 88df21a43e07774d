"""What the three fleets share (FleetCore, the one draw-materialisation kernel): the Philox streams of Fleet.noise,
RpgdFleet.draws and CemFleet.draws against a numpy restatement of Philox4x32-10 and the Box-Muller of cps_plant.cuh, the
dt refusal of cps_fleet_create, and a Philox RPGD fleet with more than 65535 experiments."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SEED = (0x2545F491 << 32) | 0x9E3779B7   # both 32-bit halves of the key non-zero
OFFSET = 5
RPGD_DRAWS_RESAMPLE, RPGD_DRAWS_RESET, CEM_DRAWS = 0xA0000000, 0xB0000000, 0xC0000000   # cps_plant.cuh


def philox4x32_10(c0, c1, c2, c3, seed):
    """Philox4x32-10 (Salmon et al., SC'11) on uint32 counters held in uint64 arrays; key = (seed low, seed high)."""
    m32 = np.uint64(0xFFFFFFFF)
    c = [np.asarray(x, dtype=np.uint64) for x in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & m32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & m32]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m32, (k1 + np.uint64(0xBB67AE85)) & m32
    return c


def box_muller(a, b):
    # the uniforms in float32 as the kernel forms them ((a >> 8) + 0.5 rounds to 24 bits), the rest in float64
    u1, u2 = ((((x >> np.uint64(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)).astype(np.float64)
              for x in (a, b))
    r = np.sqrt(-2.0 * np.log(u1))
    return r * np.cos(2.0 * np.pi * u2), r * np.sin(2.0 * np.pi * u2)


def normals(w0, w1, period, e_global, n):
    """philox_normals: n standard normals per (w0, e_global) (broadcast), four per counter (w0, w1 + group, period, e)."""
    out = []
    for g in range((n + 3) // 4):
        x, y, z, w = philox4x32_10(w0, w1 + g, period, e_global, SEED)
        out += [*box_muller(x, y), *box_muller(z, w)]
    return np.stack(out[:n], axis=-1)


def check(got, want):
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-6, atol=1e-6)


def test_fleet_noise_matches_restated_philox():
    from cartpolesimulation_b200.fleet import Fleet
    E, K, T = 3, 96, 50
    fl = Fleet(E, num_rollouts=K, horizon=T, seed=SEED, experiment_offset=OFFSET)
    assert fl.n_ind % 4 != 0
    k, e = np.arange(K)[None, :], OFFSET + np.arange(E)[:, None]
    for p in (0, 7):
        check(fl.noise(p), normals(k, 0, p, e, fl.n_ind).transpose(0, 2, 1))   # [E][n_ind][K]
    fl.close()


def test_rpgd_fleet_draws_match_restated_philox():
    from cartpolesimulation_b200.fleet import RpgdFleet
    E, K = 3, 16
    fl = RpgdFleet(E, num_rollouts=K, mpc_horizon=35, seed=SEED, experiment_offset=OFFSET)
    assert fl.n_ind % 4 != 0
    e = OFFSET + np.arange(E)[:, None]
    rows = K - fl.opt_keep_k
    for p in (0, 3):
        check(fl.draws(p), normals(np.arange(rows)[None, :], RPGD_DRAWS_RESAMPLE, p, e, fl.n_ind))   # [E][rows][n_ind]
    check(fl.draws(-1), normals(np.arange(K)[None, :], RPGD_DRAWS_RESET, 0, e, fl.n_ind))
    fl.close()


def test_cem_fleet_draws_match_restated_philox():
    from cartpolesimulation_b200.fleet import CemFleet
    E, K, T = 3, 64, 35
    assert T % 4 != 0
    fl = CemFleet(E, num_rollouts=K, mpc_horizon=T, cem_outer_it=2, cem_best_k=8, seed=SEED, experiment_offset=OFFSET)
    fl.reset(np.zeros((E, 6), np.float32), period=2)
    k, e = np.arange(K)[None, :], OFFSET + np.arange(E)[:, None]
    for p in (2, 5):
        assert fl.iterations(p) == 2
        want = np.stack([normals(k, CEM_DRAWS + it * ((T + 3) // 4), p, e, T).transpose(0, 2, 1) for it in range(2)])
        check(fl.draws(p), want)   # [it][E][T][K]
    fl.close()


def test_fleet_create_refuses_a_period_that_is_not_sim_substeps_ticks():
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    eng = Engine(64, 20, dt=0.02)
    c = L.cps_fleet_config(C.sizeof(L.cps_fleet_config), 2, 7, L.FLEET_NOISE_PHILOX, 0.002, 0, 0)
    assert eng.lib.cps_fleet_create(eng._h, C.byref(c)) == 1   # CPS_ERR_INVALID: 7 x 0.002 != 0.02
    c.sim_substeps = 10
    assert eng.lib.cps_fleet_create(eng._h, C.byref(c)) == 0
    eng.close()


def test_philox_rpgd_fleet_beyond_65535_experiments():
    from cartpolesimulation_b200.fleet import RpgdFleet
    E, K, T = 65536, 16, 10
    rng = np.random.default_rng(0)
    s = np.zeros((E, 6), np.float32)
    s[:, 0] = rng.uniform(-np.pi, np.pi, E)
    s[:, 1] = rng.uniform(-1.0, 1.0, E)
    s[:, 2], s[:, 3] = np.cos(s[:, 0]), np.sin(s[:, 0])
    s[:, 4] = rng.uniform(-0.15, 0.15, E)
    fl = RpgdFleet(E, num_rollouts=K, mpc_horizon=T, seed=SEED)
    fl.reset(s)
    fl.run(1)
    assert fl.period == 1
    assert np.isfinite(fl.states()).all()
    last = fl.draws(-1)[E - 1].clone()
    fl.close()
    one = RpgdFleet(1, num_rollouts=K, mpc_horizon=T, seed=SEED, experiment_offset=E - 1)
    assert torch.equal(last, one.draws(-1)[0])
    one.close()
