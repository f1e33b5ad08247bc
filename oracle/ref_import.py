"""Test-only helper: import the UNMODIFIED reference (eloialonso/diamond) from /root/reference/src.

ORACLE / TEST INFRASTRUCTURE ONLY.  Nothing in the product path (diamond_b200/) may import this.
The reference is not part of this repository, so this module is only used by
oracle/make_golden.py to generate the fixtures under tests/golden/; no test imports it.

The reference needs omegaconf / hydra / gymnasium / ale_py / torcheval at *import* time only
(utils.py:11, trainer.py:7, envs/env.py:4-6, models/rew_end_model.py:8); none of them is used on the
hot path, so empty stub modules are injected into sys.modules (SURVEY.md section 8c).
"""
import importlib
import os
import sys
import types

REF_SRC = os.environ.get("DIAMOND_REFERENCE_SRC", "/root/reference/src")


def available() -> bool:
    return os.path.isdir(os.path.join(REF_SRC, "models"))


def _stub(name, **attrs):
    if name in sys.modules:
        return sys.modules[name]
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    parent, _, child = name.rpartition(".")
    if parent:
        setattr(_stub(parent), child, m)
    return m


def install_stubs() -> None:
    class _Dummy:  # generic placeholder type
        def __init__(self, *a, **k):
            pass

    class _Wrapper(_Dummy):
        pass

    class _RecordCtor(_Dummy):
        pass

    for mod in ("omegaconf", "hydra", "hydra.utils", "ale_py", "wandb", "cv2"):
        try:
            importlib.import_module(mod)
        except Exception:
            _stub(mod)
    om = sys.modules["omegaconf"]
    for n in ("DictConfig", "OmegaConf"):
        if not hasattr(om, n):
            setattr(om, n, _Dummy)
    hu = sys.modules["hydra.utils"]
    if not hasattr(hu, "instantiate"):
        hu.instantiate = lambda *a, **k: None
    try:
        importlib.import_module("gymnasium")
    except Exception:
        g = _stub("gymnasium", Wrapper=_Wrapper, Env=_Dummy, ObservationWrapper=_Wrapper, make=lambda *a, **k: None)
        _stub("gymnasium.vector", AsyncVectorEnv=_Dummy)
        _stub("gymnasium.core", Env=_Dummy, WrapperActType=object, WrapperObsType=object)
        _stub("gymnasium.spaces", Box=_Dummy, Discrete=_Dummy)
        _stub("gymnasium.utils", RecordConstructorArgs=_RecordCtor)
        g.utils = sys.modules["gymnasium.utils"]
        g.spaces = sys.modules["gymnasium.spaces"]
    try:
        importlib.import_module("torcheval.metrics.functional")
    except Exception:
        _stub("torcheval")
        _stub("torcheval.metrics")
        _stub("torcheval.metrics.functional", multiclass_confusion_matrix=lambda *a, **k: None)


def load():
    """Returns a namespace with the reference modules (models, envs, agent, data, utils)."""
    if not available():
        raise RuntimeError(f"reference tree not found at {REF_SRC}")
    install_stubs()
    if REF_SRC not in sys.path:
        sys.path.insert(0, REF_SRC)
    ns = types.SimpleNamespace()
    ns.blocks = importlib.import_module("models.blocks")
    ns.diffusion = importlib.import_module("models.diffusion")
    ns.actor_critic = importlib.import_module("models.actor_critic")
    ns.rew_end_model = importlib.import_module("models.rew_end_model")
    ns.envs = importlib.import_module("envs")
    ns.agent = importlib.import_module("agent")
    ns.data = importlib.import_module("data")
    ns.utils = importlib.import_module("utils")
    ns.env_loop = importlib.import_module("coroutines.env_loop")
    return ns
