"""The reference itself, for the drop-in test and the Python CPU baseline of bench.py.

`baseline/_ref/` is a git-ignored COPY of the reference's `src/` made by `__graft_entry__.build()` when
UAVSIM_REFERENCE_SRC names a checkout of it (the reference is a plain source tree: there is nothing to pip-install).
Nothing here is imported by the product (marl_uavs_targets_tracking_b200/) -- only tests/ and bench.py use it, and both
skip cleanly when the copy is absent.
"""
import os
import shutil
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref", "src")


def sync_reference(src=None):
    """Copy the reference's src/ (default: $UAVSIM_REFERENCE_SRC) into baseline/_ref/src.  Returns the path or None."""
    src = src or os.environ.get("UAVSIM_REFERENCE_SRC")
    if not src or not os.path.isdir(src):
        return REF_DIR if os.path.isdir(REF_DIR) else None
    if os.path.isdir(REF_DIR):
        shutil.rmtree(REF_DIR)
    shutil.copytree(src, REF_DIR, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    return REF_DIR


def available():
    return os.path.isfile(os.path.join(REF_DIR, "environment.py"))


def import_reference():
    """Import the UNMODIFIED reference modules from baseline/_ref/src.  src/train.py pulls matplotlib / imageio in
    through utils.draw_util (absent in this image): that one module is stubbed (SURVEY.md section 8c), nothing else."""
    if not available():
        raise ImportError("baseline/_ref/src is missing: run __graft_entry__.build() with UAVSIM_REFERENCE_SRC set")
    sys.dont_write_bytecode = True
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    stub = types.ModuleType("utils.draw_util")
    stub.draw_animation = lambda *a, **k: None
    stub.plot_reward_curve = lambda *a, **k: None
    import utils  # noqa: F401  (the reference's package)
    sys.modules["utils.draw_util"] = stub
    for name in ("tensorboard", "torch.utils.tensorboard"):
        try:
            __import__(name)
        except Exception:
            m = types.ModuleType(name)
            m.SummaryWriter = object
            sys.modules[name] = m
    import environment as ref_environment
    import train as ref_train
    from models.PMINet import PMINetwork
    from models.actor_critic import ActorCritic
    return types.SimpleNamespace(environment=ref_environment, train=ref_train, PMINetwork=PMINetwork,
                                 ActorCritic=ActorCritic, dir=REF_DIR)


def load_yaml_config(method):
    """The reference's YAML for `method` the way main.py uses it, without args_util.get_config's side effects
    (mkdir under the reference tree, CUDA_VISIBLE_DEVICES)."""
    import yaml
    with open(os.path.join(REF_DIR, "configs", method + ".yaml"), encoding="UTF-8") as f:
        cfg = yaml.load(f, Loader=yaml.FullLoader)
    if method == "MAAC":
        cfg["cooperative"] = 0  # src/main.py:75-76
    return cfg
