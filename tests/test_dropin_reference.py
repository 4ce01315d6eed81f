"""CPU: the drop-in claim of INTEGRATION.md section A, executed against what the unmodified reference does there
(recorded by tests/golden/make_golden.py into tests/golden/dropin_reference.npz).

1. The registry / seam patch printed in INTEGRATION.md is extracted from the markdown and exec'd against stand-in modules
   carrying the reference's module paths and names; afterwards those lookups resolve to the xuance_b200 classes, and the
   reference resolves its learner through that registry.
2. The keyword arguments the reference's ``OnPolicyAgent._build_memory`` (on_policy.py:65-104) passed to the patched
   buffer class bind to the xuance_b200 buffer constructor, and the constructor runs with them (on a CPU-only machine it
   stops at the CUDA allocation - there is no CPU fallback to fall into).
3. The restatement of the reference's ``OnPolicyAgent.train_epochs`` (on_policy.py:182-205) in oracle/agents.py drives a
   recording fake with the same NumPy seed and produces the reference's call sequence.  tests/test_gpu_dropin.py then runs
   that restatement over the real xuance_b200 buffer + learner on the GPU."""
import inspect
import json
import os
import re
import sys
import types
from argparse import Namespace
from types import SimpleNamespace

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(ROOT, "tests", "golden", "dropin_reference.npz"), allow_pickle=False)


def _stand_in_reference(ref, monkeypatch):
    """Empty modules under the reference's package paths holding its registry keys and on-policy buffer names."""
    mods = {}
    for path in ref["registry/modules"]:
        parts = str(path).split(".")
        for i in range(1, len(parts) + 1):
            name = ".".join(parts[:i])
            if name not in mods:
                mods[name] = types.ModuleType(name)
                monkeypatch.setitem(sys.modules, name, mods[name])
                if i > 1:
                    setattr(mods[".".join(parts[:i - 1])], parts[i - 1], mods[name])
    mods["xuance.torch.learners"].REGISTRY_Learners = {str(k): object() for k in ref["registry/learner_names"]}
    core = mods["xuance.torch.agents.core.on_policy"]
    for name in ref["registry/on_policy_buffers"]:
        setattr(core, str(name), type(str(name), (), {}))
    return mods


def test_registry_patch_from_the_document_resolves_to_xb200(ref, monkeypatch):
    mods = _stand_in_reference(ref, monkeypatch)
    md = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    section = md[md.index("Registering inside an existing XuanCe checkout"):]
    code = re.search(r"```python\n(.*?)```", section, re.S).group(1)
    exec(compile(code, "INTEGRATION.md#A", "exec"), {})
    import xuance_b200.common as xc
    from xuance_b200.torch.learners import PPO_Learner
    core = mods["xuance.torch.agents.core.on_policy"]
    assert mods["xuance.torch.learners"].REGISTRY_Learners["PPO_Learner"] is PPO_Learner
    assert sorted(ref["registry/on_policy_buffers"]) == ["DummyOnPolicyBuffer", "DummyOnPolicyBuffer_Atari"]
    assert core.DummyOnPolicyBuffer is xc.DummyOnPolicyBuffer and core.DummyOnPolicyBuffer_Atari is xc.DummyOnPolicyBuffer_Atari
    # the reference resolves its learner through the registry at build time (agents/base/agent.py: _build_learner)
    assert bool(ref["registry/build_learner_uses_registry"])


@pytest.mark.parametrize("atari", [False, True])
def test_reference_build_memory_reaches_the_xb200_buffer(ref, atari, monkeypatch):
    import xuance_b200.common as xc
    from xuance_b200.common import Box, Discrete
    cls = xc.DummyOnPolicyBuffer_Atari if atari else xc.DummyOnPolicyBuffer
    obs_space = Box(0, 255, (84, 84, 4), np.uint8) if atari else Box(-1, 1, (4,), np.float32)
    agent = SimpleNamespace(observation_space=obs_space, action_space=Discrete(4), n_envs=4, horizon_size=8, n_minibatch=2,
                            gamma=0.99, gae_lam=0.95, is_tensor_memory=False,
                            config=Namespace(use_gae=True, use_advnorm=True, env_name="Atari" if atari else "Classic"))
    seen = json.loads(str(ref["build_memory/%s/kwargs" % atari]))
    assert seen.pop("_n_positional") == 0
    # values the reference took from the agent are recorded as "agent.<name>"
    kw = {k: getattr(agent, v[6:]) if isinstance(v, str) and v.startswith("agent.") else v for k, v in seen.items()}
    kw["auxiliary_shape"] = {k: tuple(v) for k, v in kw["auxiliary_shape"].items()}
    assert kw["observation_space"] is agent.observation_space and kw["action_space"] is agent.action_space
    inspect.signature(cls.__init__).bind(None, **kw)                     # the reference's kwargs fit the constructor
    import torch
    if torch.cuda.is_available():
        buf = cls(**kw)
        assert isinstance(buf, cls) and buf.observations.is_cuda
    else:
        with pytest.raises((RuntimeError, AssertionError)):       # CUDA allocation: no CPU fallback behind the seam
            cls(**kw)
    assert set(seen) == {"observation_space", "action_space", "auxiliary_shape", "n_envs", "horizon_size", "use_gae",
                         "use_advnorm", "gamma", "gae_lam"}
    assert list(ref["build_memory/%s/buffer_batch" % atari]) == [32, 16]


class _Recorder:
    def __init__(self):
        self.calls = []

    def sample(self, idx):
        self.calls.append(("sample", np.array(idx, copy=True)))
        return {"obs": idx[:1], "actions": idx[:1], "returns": idx[:1], "values": idx[:1], "advantages": idx[:1],
                "aux_batch": {}, "batch_size": len(idx)}

    def update(self, **samples):
        self.calls.append(("update", ",".join(sorted(samples))))
        return {"n": len(self.calls)}


@pytest.mark.parametrize("buffer_size,batch_size,n_epochs", [(64, 16, 4), (60, 16, 3)])
def test_train_epochs_restatement_equals_the_live_reference(ref, buffer_size, batch_size, n_epochs):
    from oracle.agents import reference_train_epochs
    rec = _Recorder()
    np.random.seed(11)
    info = reference_train_epochs(SimpleNamespace(buffer_size=buffer_size, batch_size=batch_size, memory=rec, learner=rec),
                                  n_epochs)
    p = "train_epochs/%d_%d_%d" % (buffer_size, batch_size, n_epochs)
    a = rec.calls
    assert info == {"n": int(ref[p + "/info_n"])} and len(a) == 2 * n_epochs * -(-buffer_size // batch_size)
    assert [k for k, _ in a] == list(ref[p + "/kinds"])
    samples = [v for k, v in a if k == "sample"]
    assert [len(v) for v in samples] == list(ref[p + "/sample_len"])
    assert np.array_equal(np.concatenate(samples), ref[p + "/sample_idx"])
    assert [v for k, v in a if k == "update"] == list(ref[p + "/update_keys"])
