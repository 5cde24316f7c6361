#!/usr/bin/env python
"""Run an UNMODIFIED driver of the reference (src/main.py, src/sl.py) on the classes of graph_marl_b200.

    python tools/run_reference_driver.py main.py --env-type=simple --model=dqn --netmon ... --device=cuda
    GM_DEFAULT_DEVICE=cuda python tools/run_reference_driver.py sl.py --iterations 200 ...      # sl.py has no --device

The drivers are executed from an unedited copy of the reference's src/ (baseline/_ref/src, git-ignored and not part of
this repository, or $GM_REFERENCE_SRC).  Before the driver starts, the modules it imports for the
hot path are aliased in sys.modules to this package -- the import swap INTEGRATION.md section 2 describes:

    env.network / env.routing / env.simple_environment / env.wrapper / env.environment / env.constants,
    replaybuffer, buffer          -> graph_marl_b200.*
    model    : NetMon, DQN, MLP   -> graph_marl_b200.model (DGN, DQNR, CommNet stay the reference's)
    policy   : EpsilonGreedy      -> graph_marl_b200.policy (ShortestPath, RandomPolicy, SimplePolicy stay the reference's)

eval.py, util.py and the driver itself are the reference's own files.  The three packages the reference imports that
are not in this image (gymnasium, matplotlib, torch_geometric: plotting / non-default aggregations only) are stubbed
by tools/ref_stubs.py.
"""
import importlib
import os
import runpy
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF_SRC = os.environ.get("GM_REFERENCE_SRC", os.path.join(ROOT, "baseline", "_ref", "src"))


def install_aliases():
    sys.path.insert(0, HERE)
    sys.path.insert(0, ROOT)
    import ref_stubs

    ref_stubs.REFERENCE_SRC = REF_SRC
    ref_stubs.install()
    if REF_SRC not in sys.path:
        sys.path.insert(0, REF_SRC)
    # the reference's own modules that are NOT on the hot path, imported under private names first
    ref_model = importlib.import_module("model")
    ref_policy = importlib.import_module("policy")
    for name in ("env", "env.network", "env.routing", "env.simple_environment", "env.wrapper", "env.environment",
                 "env.constants", "replaybuffer", "buffer", "model", "policy"):
        sys.modules.pop(name, None)

    import graph_marl_b200.buffer as gm_buffer
    import graph_marl_b200.env as gm_env
    import graph_marl_b200.model as gm_model
    import graph_marl_b200.policy as gm_policy
    import graph_marl_b200.replaybuffer as gm_replay

    sys.modules["env"] = gm_env
    for sub in ("network", "routing", "simple_environment", "wrapper", "environment", "constants"):
        sys.modules["env." + sub] = importlib.import_module("graph_marl_b200.env." + sub)
    sys.modules["replaybuffer"] = gm_replay
    sys.modules["buffer"] = gm_buffer
    model = types.ModuleType("model")
    model.__dict__.update({k: v for k, v in ref_model.__dict__.items() if not k.startswith("__")})
    for k in ("NetMon", "DQN", "MLP", "Q_Net", "SimpleAggregation"):
        setattr(model, k, getattr(gm_model, k))
    sys.modules["model"] = model
    policy = types.ModuleType("policy")
    policy.__dict__.update({k: v for k, v in ref_policy.__dict__.items() if not k.startswith("__")})
    policy.EpsilonGreedy = gm_policy.EpsilonGreedy
    sys.modules["policy"] = policy


def main():
    if len(sys.argv) < 2:
        raise SystemExit(__doc__)
    driver = os.path.join(REF_SRC, sys.argv[1])
    if not os.path.exists(driver):
        raise SystemExit(f"{driver} is missing: copy the src/ directory of jw3il/graph-marl to {REF_SRC}")
    install_aliases()
    if os.environ.get("GM_DEFAULT_DEVICE"):
        # sl.py has no --device flag: it builds its tensors on torch's default device (the CPU); this package has no CPU
        # path, so the launcher moves the default device instead of editing the driver
        import torch

        torch.set_default_device(os.environ["GM_DEFAULT_DEVICE"])
    sys.argv = [driver] + sys.argv[2:]
    runpy.run_path(driver, run_name="__main__")


if __name__ == "__main__":
    main()
