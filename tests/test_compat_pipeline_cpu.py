"""The shipped vectorisation boundary (SURVEY 8(b)): compat/core/rl_framework/utils/pipeline.py serves
``ReinforcementLearningPipeline.create_vectorized_environment`` (reference pipeline.py:32-61,64-119) at the reference's
module paths -- the current ``core.rl_framework`` and the ``threatengage.rl_framework`` the apps still import -- without
hiding the rest of the reference's packages.  Runs in a fresh interpreter with stand-ins for the third-party packages
the test environment lacks (tests/_stub_modules.py).  A stand-in of the reference's package layout, written by the test,
checks that compat inherits and re-exports the reference's own members; the env-construction path of the reference's own
training app apps/threatengage_runner/stage03/experiments/02/bo_exp02_vFinal_home_office_app.py is executed unmodified
when DRONECHASE_REFERENCE names a checkout of the reference."""
import json
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.abspath(os.environ["DRONECHASE_REFERENCE"]) if os.environ.get("DRONECHASE_REFERENCE") else ""


def _run(code, extra_path=()):
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "compat"), *extra_path, ROOT, os.path.join(ROOT, "tests")])
    env["DRONECHASE_B200_ENVS"] = "4096"
    out = subprocess.run([sys.executable, "-c", textwrap.dedent(code)], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


PRELUDE = """
import json, sys
import _stub_modules; _stub_modules.install()
import dronechase_b200.vec_env as ve
made = []
class FakeVecEnv:                      # stands in for the CUDA-backed DroneChaseVecEnv (no GPU in the CPU suite)
    def __init__(self, cfg, n_envs=8, seed=0, device=0, **kw):
        self.cfg, self.num_envs = cfg, n_envs
        self.action_space = self.observation_space = None
        made.append(self)
ve.DroneChaseVecEnv = FakeVecEnv
"""


def test_pipeline_without_the_reference_on_the_path():
    r = _run(PRELUDE + """
from core.rl_framework.utils.pipeline import ReinforcementLearningPipeline as P1
from threatengage.rl_framework.utils.pipeline import ReinforcementLearningPipeline as P2
from threatengage.environments.level4.exp03_vFinal_environment import Exp03vFinalEnvironment
from threatsense.level5.level5_c1_fusion_environment import Level5C1FusionEnvironment
from core.rl_framework.utils.io_data import MultiH5Dataset
kw = {"rl_frequency": 30, "dome_radius": 25, "learning_rate": 1e-4}
a = P1.create_vectorized_environment(Exp03vFinalEnvironment, env_kwargs=kw)
b = P2.create_vectorized_multi_agent_v2_environment(Level5C1FusionEnvironment, {}, n_envs=12)
assert kw == {"rl_frequency": 30, "dome_radius": 25, "learning_rate": 1e-4}     # the caller's dict is not edited
print(json.dumps({"mon": [type(a).__name__, type(b).__name__], "n": [m.num_envs for m in made],
                  "cfg": [[m.cfg.n_lw, m.cfg.n_lm, m.cfg.rl_frequency, m.cfg.dome_radius, m.cfg.family] for m in made],
                  "wrapped": a.venv is made[0]}))
""")
    assert r["mon"] == ["VecMonitor", "VecMonitor"] and r["wrapped"]
    assert r["n"] == [4096, 12]                                             # DRONECHASE_B200_ENVS / explicit n_envs
    assert r["cfg"][0] == [2, 9, 30, 25.0, "stage03"] and r["cfg"][1][4] == "level5"


@pytest.mark.skipif(not REF or not os.path.isdir(REF), reason="DRONECHASE_REFERENCE does not name a checkout of the reference")
def test_reference_training_app_builds_its_vec_env_unchanged():
    r = _run(PRELUDE + """
import importlib.util, os
ref = os.path.abspath(os.environ["DRONECHASE_REFERENCE"])
# the rest of the reference's packages stays importable behind compat/ (extend_path), e.g. the directory manager and
# the navigators; compat only shadows the env modules, pipeline.py and io_data.py
from core.rl_framework.utils.directory_manager import DirectoryManager
import core.entities.navigators.geometry_utils as gu
import core.rl_framework.utils.pipeline as pl
spec = importlib.util.spec_from_file_location(
    "bo_app", os.path.join(ref, "apps/threatengage_runner/stage03/experiments/02/bo_exp02_vFinal_home_office_app.py"))
app = importlib.util.module_from_spec(spec); spec.loader.exec_module(app)            # the app, unmodified
suggestions = {"rl_frequency": 15, "learning_rate": 1e-4, "batch_size": 512, "hidden_1": 128}
venv = app.ReinforcementLearningPipeline.create_vectorized_environment(environment=app.level4, env_kwargs=suggestions)
m = made[0]
print(json.dumps({"ref_loaded": pl._ref is not None, "has_ref_members": hasattr(app.ReinforcementLearningPipeline, "create_callback_list"),
                  "callbacklist": hasattr(app, "callbacklist") and hasattr(app, "CallbackType"),
                  "dm": DirectoryManager.__module__, "gu": gu.__file__.startswith(ref),
                  "env": app.level4.__module__, "n": m.num_envs, "cfg": [m.cfg.n_lw, m.cfg.n_lm, m.cfg.rl_frequency],
                  "mon": type(venv).__name__, "mon_mod": type(venv).__module__}))
""", extra_path=(os.path.join(REF, "src"),))
    assert r["ref_loaded"] and r["has_ref_members"] and r["callbacklist"]
    assert r["dm"].endswith("directory_manager") and r["gu"]
    assert r["env"] == "dronechase_b200.gym_env" and r["n"] == 4096 and r["cfg"] == [1, 6, 15]
    assert r["mon"] == "VecMonitor" and r["mon_mod"].startswith("stable_baselines3")      # the (stubbed) SB3 class


# a stand-in of the reference's src/ with the members compat must keep: its own pipeline module (SB3 vectorisation,
# callbacklist / CallbackType, create_callback_list) and packages compat does not shadow at all
STAND_IN_SRC = {
    "core/rl_framework/utils/pipeline.py": """
        from enum import Enum
        from stable_baselines3.common.vec_env import SubprocVecEnv, VecMonitor
        class CallbackType(Enum):
            EVAL = 1
        def callbacklist(*callbacks):
            return list(callbacks)
        class ReinforcementLearningPipeline:
            @staticmethod
            def create_vectorized_environment(environment, env_kwargs={}, n_envs=4, GUI=False, env_args=None):
                return VecMonitor(SubprocVecEnv([lambda: environment(**env_kwargs)] * n_envs))
            @staticmethod
            def create_callback_list(*callbacks):
                return callbacklist(*callbacks)
        """,
    "core/rl_framework/utils/directory_manager.py": "class DirectoryManager:\n    pass\n",
    "core/entities/__init__.py": "",
    "core/entities/navigators/__init__.py": "",
    "core/entities/navigators/geometry_utils.py": "def angle_between(a, b):\n    return 0.0\n",
}


def test_stand_in_reference_members_stay_behind_compat(tmp_path):
    src = tmp_path / "src"
    for rel, text in STAND_IN_SRC.items():
        (src / rel).parent.mkdir(parents=True, exist_ok=True)
        (src / rel).write_text(textwrap.dedent(text))
    r = _run(PRELUDE + """
from core.rl_framework.utils.directory_manager import DirectoryManager
import core.entities.navigators.geometry_utils as gu
import core.rl_framework.utils.pipeline as pl
# the import lines of the apps (threatengage.rl_framework path) and the env class of the exp02 training app
from threatengage.rl_framework.utils.pipeline import ReinforcementLearningPipeline, callbacklist, CallbackType
from threatengage.environments.level4.exp02_vFinal_environment import Exp02vFinalEnvironment as level4
suggestions = {"rl_frequency": 15, "learning_rate": 1e-4, "batch_size": 512, "hidden_1": 128}
venv = ReinforcementLearningPipeline.create_vectorized_environment(environment=level4, env_kwargs=suggestions)
class OtherEnv:                        # not a dronechase_b200 facade: the reference's own SB3 path serves it
    pass
other = ReinforcementLearningPipeline.create_vectorized_environment(OtherEnv, n_envs=3)
m = made[0]
print(json.dumps({"ref_loaded": pl._ref is not None, "same_class": ReinforcementLearningPipeline is pl.ReinforcementLearningPipeline,
                  "callback_list": ReinforcementLearningPipeline.create_callback_list(1, 2), "callback_type": CallbackType.EVAL.value,
                  "callbacklist_is_ref": callbacklist is pl._ref.callbacklist,
                  "dm": DirectoryManager.__module__, "gu": gu.__file__,
                  "env": level4.__module__, "n": m.num_envs, "cfg": [m.cfg.n_lw, m.cfg.n_lm, m.cfg.rl_frequency],
                  "mon": type(venv).__name__, "mon_mod": type(venv).__module__, "wrapped": venv.venv is m,
                  "other": [type(other).__name__, type(other.args[0]).__name__, len(other.args[0].args[0]), len(made)]}))
""", extra_path=(str(src),))
    assert r["ref_loaded"] and r["same_class"] and r["callback_list"] == [1, 2] and r["callback_type"] == 1 and r["callbacklist_is_ref"]
    assert r["dm"] == "core.rl_framework.utils.directory_manager" and os.path.realpath(r["gu"]).startswith(os.path.realpath(src))
    assert r["env"] == "dronechase_b200.gym_env" and r["n"] == 4096 and r["cfg"] == [1, 6, 15]
    assert r["mon"] == "VecMonitor" and r["mon_mod"].startswith("stable_baselines3") and r["wrapped"]
    assert r["other"] == ["VecMonitor", "SubprocVecEnv", 3, 1]          # no GPU batch was made for it


def test_fallback_vec_monitor_contract():
    import numpy as np
    from dronechase_b200.vec_env import InfoList
    from dronechase_b200.vec_monitor import VecMonitor

    class Toy:
        num_envs, observation_space, action_space = 3, None, None
        t = 0
        def reset(self): return {"x": np.zeros(3)}
        def step_async(self, a): self.a = a
        def step_wait(self):
            self.t += 1
            done = np.array([self.t % 2 == 0, False, self.t % 3 == 0])
            info = np.zeros((3, 8), dtype=np.int32); info[:, 0] = self.t
            return {"x": np.zeros(3)}, np.array([1.0, 2.0, 3.0], np.float32), done, InfoList(info, {})
        def close(self): self.closed = True
        cfg = "toy"

    m = VecMonitor(Toy())
    m.reset()
    eps = []
    for _ in range(6):
        _, _, dones, infos = m.step(np.zeros((3, 4)))
        assert len(infos) == 3
        for i in np.nonzero(dones)[0]:
            eps.append((int(i), infos[int(i)]["episode"]["r"], infos[int(i)]["episode"]["l"], infos[int(i)]["agent_kills"]))
        assert all("episode" not in infos[int(i)] for i in np.nonzero(~dones)[0])
    assert eps == [(0, 2.0, 2, 2), (2, 9.0, 3, 3), (0, 2.0, 2, 4), (0, 2.0, 2, 6), (2, 9.0, 3, 6)]
    assert m.cfg == "toy" and m.episode_count == 5
    m.close()
