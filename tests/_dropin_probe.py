"""Runs in a subprocess of tests/test_reference_dropin.py (needs the reference checkout at CPS_REFERENCE_ROOT).

Drives the UNMODIFIED reference controller_mpc in a scratch workspace (SURVEY Appendix B.10) whose
config selects `optimizer: mppi-b200`; the plugin stub is found by the reference's own glob.  There is no GPU
here, so cartpolesimulation_b200's Engine is replaced by a recorder: the probe checks everything the optimizer
extracts from the reference's wrapper objects and how it drives the C-ABI layer, not the arithmetic.
Prints one JSON object."""
import json
import os
import shutil
import sys
import tempfile

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import numpy as np  # noqa: E402
import yaml  # noqa: E402

from oracle import ref_loader as R  # noqa: E402
from tests.dropin_recorder import recording_engine  # noqa: E402


def main():
    ws = tempfile.mkdtemp(prefix="cps_dropin_")
    try:
        for d in ("Control_Toolkit_ASF", "SI_Toolkit_ASF"):
            shutil.copytree(os.path.join(R.REF, d), os.path.join(ws, d))
        shutil.copy(os.path.join(R.REF, "cartpole_physical_parameters.yml"), ws)
        # the application-specific optimizer folder does not exist in the reference checkout: create it as a package
        odir = os.path.join(ws, "Control_Toolkit_ASF", "Optimizers")
        os.makedirs(odir, exist_ok=True)
        open(os.path.join(odir, "__init__.py"), "a").close()
        shutil.copy(os.path.join(REPO, "cartpolesimulation_b200", "dropin", "Control_Toolkit_ASF", "Optimizers",
                                 "optimizer_mppi_b200.py"), odir)
        pc = os.path.join(ws, "Control_Toolkit_ASF", "config_controllers.yml")
        cc = yaml.safe_load(open(pc))
        cc["mpc"].update(optimizer="mppi-b200", predictor_specification="ODE",
                         cost_function_specification="quadratic_boundary_grad_minimal",
                         computation_library="pytorch", device="cpu", controller_logging=False)
        yaml.safe_dump(cc, open(pc, "w"))
        po = os.path.join(ws, "Control_Toolkit_ASF", "config_optimizers.yml")
        co = yaml.safe_load(open(po))
        co["mppi-b200"] = dict(co["mppi"], seed=3, mpc_horizon=50, num_rollouts=2000)
        yaml.safe_dump(co, open(po, "w"))
        pf = os.path.join(ws, "Control_Toolkit_ASF", "config_cost_function.yml")
        cf = yaml.safe_load(open(pf))
        cf["CartPole"]["quadratic_boundary_grad_minimal"]["ep_weight_up"] = 41.5   # must reach the kernel parameters
        yaml.safe_dump(cf, open(pf, "w"))

        R.load(workdir=ws)
        # predictor_ODE defaults to TensorFlowLibrary when the wrapper does not forward the library (B.10)
        import SI_Toolkit.Predictors.predictor_ODE as pode
        from SI_Toolkit.computation_library import PyTorchLibrary
        _init = pode.predictor_ODE.__init__
        pode.predictor_ODE.__init__ = lambda self, *a, **k: _init(self, *a, **dict(k, computation_library=PyTorchLibrary()))

        calls = []
        import cartpolesimulation_b200.optimizer_mppi_b200 as mod
        mod.Engine = recording_engine(calls)

        from Control_Toolkit.Controllers.controller_mpc import controller_mpc
        ctrl = controller_mpc(environment_name="CartPole",
                              control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)),
                              initial_environment_attributes={"target_position": 0.0, "target_equilibrium": 1.0,
                                                              "L": 0.395, "m_pole": 0.087})
        ctrl.configure()
        opt = ctrl.optimizer
        s = np.array([3.1, 0.1, np.cos(3.1), np.sin(3.1), 0.01, 0.0], dtype=np.float32)
        u1 = ctrl.step(s, 0.0, {"target_position": 0.1, "target_equilibrium": -1.0, "L": 0.3, "m_pole": 0.1})
        u2 = ctrl.step(s, 0.02, {})
        ctrl.controller_reset()
        out = dict(optimizer_class=type(opt).__name__, optimizer_module=type(opt).__module__,
                   optimizer_name=opt.optimizer_name, num_rollouts=opt.num_rollouts, mpc_horizon=opt.mpc_horizon,
                   u1=float(u1), u2=float(u2), u_type=type(u1).__name__, calls=calls,
                   predictor_class=type(ctrl.predictor).__module__, cost_class=type(ctrl.cost_function).__module__)
        print("PROBE_JSON " + json.dumps(out))
    finally:
        os.chdir(REPO)
        shutil.rmtree(ws, ignore_errors=True)


if __name__ == "__main__":
    main()
