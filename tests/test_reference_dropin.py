"""Drop-in checks of optimizer_mppi_b200 behind the reference's controller_mpc.

test_controller_mpc_inputs_drive_the_plugin replays what controller_mpc hands the plugin (tests/golden/
dropin_controller_mpc.json: constructor keywords, configure() arguments, predictor and cost-function configuration, the
variable parameters of every step) through plain stand-ins, in controller_mpc's call order, and runs everywhere.
test_reference_controller_mpc_drives_the_plugin runs the UNMODIFIED reference controller_mpc itself (tests/_dropin_probe.py)
and needs a CartPoleSimulation checkout, which the repository does not contain: it runs where CPS_REFERENCE_ROOT names
one and skips elsewhere.  Both replace the C-ABI Engine by the recorder of tests/dropin_recorder.py and make the same
assertions on what reaches it."""
import glob
import importlib.util
import json
import os
import subprocess
import sys
import types

import pytest

from tests.dropin_recorder import check_record, recording_engine

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE = os.environ.get("CPS_REFERENCE_ROOT")


def _import_optimizer_by_name(name):
    """The reference's discovery (Control_Toolkit/others/globals_and_utils.py:89-119): the file
    Control_Toolkit_ASF/Optimizers/optimizer_<name>.py holds the class optimizer_<name>; here the plugin stub shipped
    for that folder."""
    mod_name = "optimizer_" + name.replace("-", "_")
    files = glob.glob(os.path.join(REPO, "cartpolesimulation_b200", "dropin", "Control_Toolkit_ASF", "Optimizers",
                                   mod_name + ".py"))
    assert len(files) == 1, files
    spec = importlib.util.spec_from_file_location("Control_Toolkit_ASF.Optimizers." + mod_name, files[0])
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return getattr(mod, mod_name)


class _VariableParameters:
    """SI_Toolkit/General/variable_parameters.py: attributes held as 0-d tensors of the computation library."""

    def set_attributes(self, attrs):
        import torch
        for k, v in attrs.items():
            setattr(self, k, torch.tensor(v, dtype=torch.float32))


class _CostFunctionWrapper:
    """The attributes of Control_Toolkit/Cost_Functions/cost_function_wrapper.py the plugin reads: the plugin name, the
    plugin object with its YAML block in .config, and the shared variable parameters."""

    def __init__(self, d, vp):
        self.cost_function_name = d["cost_function_name"]
        self.cost_function = types.SimpleNamespace(config=dict(d["config"]), variable_parameters=vp)
        self.variable_parameters = vp

    def update_cost_parameters_from_config(self):   # controller_mpc.step calls it every tick; no reload here
        pass


def test_controller_mpc_inputs_drive_the_plugin(monkeypatch):
    import cartpolesimulation_b200.optimizer_mppi_b200 as impl
    with open(os.path.join(REPO, "tests", "golden", "dropin_controller_mpc.json")) as f:
        g = json.load(f)
    calls = []
    monkeypatch.setattr(impl, "Engine", recording_engine(calls))
    cls = _import_optimizer_by_name(g["optimizer_name"])
    c = g["controller"]
    # controller_mpc.__init__ / configure (:42-92): variable parameters, wrappers, optimizer, optimizer.configure
    vp = _VariableParameters()
    vp.set_attributes(c["initial_environment_attributes"])
    predictor = types.SimpleNamespace(predictor_type=g["predictor"]["predictor_type"],
                                      predictor_config=dict(g["predictor"]["predictor_config"]),
                                      predictor=types.SimpleNamespace())
    cost = _CostFunctionWrapper(g["cost_function"], vp)
    opt = cls(predictor=predictor, cost_function=cost, control_limits=tuple(c["control_limits"]),
              optimizer_logging=c["optimizer_logging"], computation_library=None,
              calculate_optimal_trajectory=c["calculate_optimal_trajectory"], **g["optimizer_config"])
    opt.configure(**g["configure"])
    # controller_mpc.step (:102-109): reload cost parameters, update attributes, optimizer.step
    us = []
    for st in g["steps"]:
        cost.update_cost_parameters_from_config()
        vp.set_attributes(st["updated_attributes"])
        us.append(opt.step(st["s"], st["time"]))
    opt.optimizer_reset()   # controller_reset
    r = dict(optimizer_name=opt.optimizer_name, num_rollouts=opt.num_rollouts, mpc_horizon=opt.mpc_horizon,
             u1=float(us[0]), u_type=type(us[0]).__name__, calls=calls)
    assert type(opt).__name__ == "optimizer_mppi_b200"
    check_record(r)


@pytest.mark.skipif(not (REFERENCE and os.path.isdir(os.path.join(REFERENCE, "Control_Toolkit"))),
                    reason="reference tree not present (set CPS_REFERENCE_ROOT to a CartPoleSimulation checkout)")
def test_reference_controller_mpc_drives_the_plugin():
    out = subprocess.run([sys.executable, os.path.join(REPO, "tests", "_dropin_probe.py")], capture_output=True,
                         text=True, timeout=300)
    line = [l for l in out.stdout.splitlines() if l.startswith("PROBE_JSON ")]
    assert line, out.stdout[-2000:] + out.stderr[-3000:]
    r = json.loads(line[0][len("PROBE_JSON "):])
    # discovered by the reference's glob + import_module, constructed and configured by the reference's controller_mpc
    assert r["optimizer_class"] == "optimizer_mppi_b200" and r["optimizer_name"] == "mppi-b200"
    assert r["predictor_class"].startswith("SI_Toolkit.") and r["cost_class"].startswith("Control_Toolkit.")
    check_record(r)
