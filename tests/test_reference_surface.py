"""Static check that the call surface the original project's workers/trainer.py and workers/evaluator.py use on the hot-path modules
exists in this package with compatible signatures (SURVEY.md section 8b).  The original project's sources are not part of this
repository: the check that parses them reads the tree AVDDPG_REFERENCE_ROOT names (oracle/ref_import.py) and skips without it.
Nothing is executed -- the sources are parsed and every `module.attr` access / call on environment, noise, replaybuffer, model,
ddpgagent and federated is looked up in the avddpg_b200 counterpart, and every keyword the reference passes must be accepted.
The object surface those calls return is checked without the reference.  The dynamic counterpart is tests/test_gpu_dropin.py."""
import ast
import inspect
import os

import pytest

from oracle.ref_import import REFERENCE_ROOT as REF

needs_reference = pytest.mark.skipif(not os.path.isdir(REF), reason="the original project's sources are not present "
                                     "(point AVDDPG_REFERENCE_ROOT at a checkout of it)")

MODULES = {"environment": "avddpg_b200.environment", "noise": "avddpg_b200.noise", "replaybuffer": "avddpg_b200.replaybuffer",
           "model": "avddpg_b200.model", "ddpgagent": "avddpg_b200.ddpgagent", "federated": "avddpg_b200.server.federated"}


def _calls(path):
    tree = ast.parse(open(path).read())
    found = []
    for node in ast.walk(tree):
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and isinstance(node.func.value, ast.Name) \
                and node.func.value.id in MODULES:
            found.append((node.func.value.id, node.func.attr, len(node.args), [k.arg for k in node.keywords if k.arg]))
    return found


@needs_reference
@pytest.mark.parametrize("src", ["workers/trainer.py", "workers/evaluator.py"])
def test_module_level_calls_exist_and_accept_the_reference_arguments(src):
    import importlib
    calls = _calls(os.path.join(REF, src))
    assert calls, "no hot-path calls found: the parser is broken"
    for mod, attr, n_pos, kws in calls:
        m = importlib.import_module(MODULES[mod])
        assert hasattr(m, attr), f"{src}: {mod}.{attr} has no counterpart in {MODULES[mod]}"
        target = getattr(m, attr)
        sig = inspect.signature(target.__init__ if inspect.isclass(target) else target)
        params = [p for p in sig.parameters.values() if p.name != "self"]
        names = {p.name for p in params}
        has_var_kw = any(p.kind is inspect.Parameter.VAR_KEYWORD for p in params)
        for k in kws:
            assert k in names or has_var_kw, f"{src}: {mod}.{attr}(... {k}=...) is not accepted by {MODULES[mod]}.{attr}{sig}"
        n_positional = sum(p.kind in (inspect.Parameter.POSITIONAL_ONLY, inspect.Parameter.POSITIONAL_OR_KEYWORD) for p in params)
        assert n_pos <= n_positional or any(p.kind is inspect.Parameter.VAR_POSITIONAL for p in params), \
            f"{src}: {mod}.{attr} is called with {n_pos} positional arguments, {MODULES[mod]}.{attr}{sig} takes {n_positional}"


def test_object_surface_used_by_the_trainer():
    """Attributes / methods the trainer and evaluator touch on the objects those calls return."""
    from avddpg_b200 import environment, model, noise, replaybuffer
    from avddpg_b200.server import federated
    for name in ("reset", "step", "get_jerk", "render", "close_render", "followers", "num_states", "num_actions", "hidden_multiplier",
                 "num_models", "def_num_states", "def_num_actions", "number_of_reward_components", "state_lbs", "jerk_lb", "exog_lbl"):
        assert name in dir(environment.Platoon) or name in inspect.getsource(environment.Platoon.__init__), name
    for name in ("add", "sample", "buffer_counter"):
        assert name in dir(replaybuffer.ReplayBuffer) or name in inspect.getsource(replaybuffer.ReplayBuffer.__init__), name
    for name in ("__call__", "reset"):
        assert hasattr(noise.OUActionNoise, name)
    for cls in (model.Actor, model.Critic):
        for name in ("__call__", "weights", "trainable_variables", "get_weights", "set_weights", "save"):
            assert hasattr(cls, name), (cls, name)
    for name in ("get_avg_params", "get_weighted_avg_params"):
        assert hasattr(federated.Server, name)
    from avddpg_b200 import optimizers, trainer
    assert hasattr(optimizers.Adam, "apply_gradients") and hasattr(trainer.Trainer, "learn")
