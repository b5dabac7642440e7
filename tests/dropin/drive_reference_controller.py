"""TEST-ONLY driver (run as a subprocess by tests/test_dropin_reference.py; needs the Control_Toolkit checkout named by CTK_REFERENCE).

Enters the refharness workspace (``Control_Toolkit -> $CTK_REFERENCE`` + a working ``Control_Toolkit_ASF``), copies the shim files of
``integration/Control_Toolkit_ASF/Optimizers/`` next to the application's optimizers exactly as INTEGRATION.md section 2 tells a
maintainer to, and drives the reference's UNMODIFIED ``controller_mpc`` (reference Controllers/controller_mpc.py:24-109) with
``optimizer_name="<name>-b200"``: discovery by file / class name (others/globals_and_utils.py:103-133), construction with the
controller's kwargs (:56-65), the reference's own PredictorWrapper / CostFunctionWrapper configure (:67-82), then
``optimizer.configure(dt=, predictor_specification=, num_states=, num_control_inputs=)`` (:84-89), which reaches ``ctk_create``.
Prints one JSON line per optimizer."""
import json
import os
import shutil
import sys

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, REPO)


def main():
    import numpy as np
    import yaml
    from oracle.gen_golden import CASES
    from oracle.refharness.workspace import enter_workspace
    ws = enter_workspace()
    shim_dir = os.path.join(REPO, "integration", "Control_Toolkit_ASF", "Optimizers")
    dst = os.path.join(ws, "Control_Toolkit_ASF", "Optimizers")
    os.makedirs(dst, exist_ok=True)
    for f in os.listdir(shim_dir):
        if f.endswith(".py"):
            shutil.copy(os.path.join(shim_dir, f), os.path.join(dst, f))
    import logging
    logging.disable(logging.INFO)
    from control_toolkit_b200._lib import BackendUnavailable
    results = []
    for name, fixture in (("mppi-b200", "mppi_c1_n2000"), ("cem-tf-b200", "cem_c2_n4096_k64"), ("rpgd-b200", "rpgd_c3"),
                          ("random-action-tf-b200", "random_action_n512"), ("gradient-tf-b200", "gradient_n40"),
                          ("cem-naive-grad-tf-b200", "gradcem_naive_n200"), ("cem-grad-bharadhwaj-tf-b200", "gradcem_bharadhwaj_n32")):
        base, pred_spec, cost_name, cfg, _, _ = CASES[fixture]
        cc = dict(mpc=dict(optimizer=name, predictor_specification=pred_spec, cost_function_specification=cost_name,
                           computation_library="pytorch", device="cpu", controller_logging=False, calculate_optimal_trajectory=False))
        with open(os.path.join("Control_Toolkit_ASF", "config_controllers.yml"), "w") as f:
            yaml.safe_dump(cc, f)
        from Control_Toolkit.Controllers import controller_mpc as cm  # the reference module, unmodified
        cm.config_optimizers[name] = dict(cfg)  # "copy the mppi / cem-tf / rpgd block under the new key, unchanged"
        ctrl = cm.controller_mpc(environment_name="CartPole",
                                 control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)),
                                 initial_environment_attributes={"target_position": 0.0, "target_equilibrium": 1.0})
        rec = {"optimizer": name}
        try:
            ctrl.configure(optimizer_name=name, predictor_specification=pred_spec)
            rec["outcome"] = "configured"
            u = ctrl.step(np.array([0.1, 0.0, np.cos(0.1), np.sin(0.1), 0.0, 0.0], np.float32), time=0.0)
            rec["u"] = [float(x) for x in np.ravel(u)]
            ctrl.controller_reset()
        except BackendUnavailable as e:  # raised by ctk_create on a box without a GPU: every layer above it has run
            rec["outcome"] = "backend_unavailable"
            rec["error"] = str(e)
        opt = ctrl.optimizer
        rec["class"] = type(opt).__name__
        rec["module_file"] = os.path.relpath(sys.modules[type(opt).__module__].__file__, ws)
        rec["bases"] = [b.__module__ + "." + b.__name__ for b in type(opt).__mro__[1:3]]
        rec["num_rollouts"], rec["mpc_horizon"] = int(opt.num_rollouts), int(opt.mpc_horizon)
        rec["yaml_num_rollouts"], rec["yaml_mpc_horizon"] = int(cfg["num_rollouts"]), int(cfg["mpc_horizon"])
        rec["predictor_is_reference_wrapper"] = type(opt.predictor).__module__.startswith("SI_Toolkit")
        rec["cost_is_reference_wrapper"] = type(opt.cost_function).__module__.startswith("Control_Toolkit.")
        rec["num_states"], rec["num_control_inputs"] = opt.num_states, opt.num_control_inputs
        results.append(rec)
    print("DROPIN_RESULT " + json.dumps(results))


if __name__ == "__main__":
    main()
