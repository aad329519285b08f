"""Drop-in mirror of the reference's Trainer (PKG/trainer.py:19-303) whose hot loop is a batched device driver.

`Trainer(...)` keeps the reference's positional/keyword signature and defaults (PKG/trainer.py:20-44) and adds
keyword-only extras (`num_envs`, `num_populations`, `device`, `chunk_steps`, `transfer_mode`, platform/dynamics
parameters).  `curriculum_training()` replaces the Python `for episode: while not done:` loop (PKG/trainer.py:
169-245) by `Engine.train(chunk_steps)` launches: the select -> step -> update -> auto-reset -> promotion -> transfer
cycle runs inside one CUDA kernel for all envs (csrc/train_kernel.cuh: train_kernel); the host only reads the
320-byte population state between launches to log, checkpoint and stop.

`max_num_episodes` keeps its per-env meaning (PKG/trainer.py:190: one env runs at most that many episodes per curriculum
step, and epsilon is a function of that env's episode index, :112-126): with N envs sharing the agent the device counts
finished episodes pooled over all of them, so the limit handed to it is `max_num_episodes * N` -- the forced advance
comes when the MEAN per-env episode index reaches `max_num_episodes`, and N = 1 is the reference.  The logged episode
index, remaining episodes and exploration rate are per-env figures (pooled count // N).
"""
from __future__ import annotations

import math
import pickle
from collections import deque
from datetime import datetime
from pathlib import Path
from typing import Any, Dict, Optional, Sequence

import numpy as np

from . import ASSETS_PATH
from . import constants as K
from .double_q_learning import DoubleQLearningAgent, StateAction

_TIME_FORMAT = r"%d-%m-%Y %H:%M:%S"


def replica_shape(num_envs: int, merge_every: int = 1) -> int:
    """Envs per replica for ONE agent on `num_envs` envs (replica-merge mode, DESIGN.md section 3).  Merging after every step the
    merge grows with the number of replicas while a replica's step grows with its envs: about 128 replicas is the measured optimum
    on a B200 up to 1,024 envs per replica (65,536 envs: 128 x 512 envs 15.3 us per step, 512 x 128 18.6, 64 x 1,024 18.9; 262,144
    envs: 256 x 1,024 24.1, 128 x 2,048 28.1, 512 x 512 32.0; profiles/r02_coop_merge_rejected.txt), and the learning curve does not depend on the split (tools/learn_probe.py:
    0.814 / 0.815 after 2,700 episodes per env for 64, 128 and 512 replicas).  With rarer merges more, smaller replicas win
    (every 16 steps: 512 x 128 5.0 us per step, 128 x 512 7.3)."""
    if merge_every > 1:
        return 128
    per = -(-num_envs // 128)
    return min(max(-(-per // 128) * 128, 128), 1024)


class Trainer:
    _eval_every: Optional[int] = None       # greedy evaluation of every agent after each `eval_every`-th chunk (None: off)
    _eval_episodes: int = 1024
    _eval_two_axis: Optional[K.TwoAxisParameters] = None      # also the two-axis landing (x policy on x, its mirror on y)
    _eval_platforms: Optional[list] = None      # also the landing under each of these (r_mp, v_mp) platform motions

    def __init__(
        self,
        curriculum_steps: int = 5,
        double_q_learning_agent: Optional[DoubleQLearningAgent] = None,
        successive_successful_episodes: int = 100,
        success_rate: float = 0.96,
        max_num_episodes: int = 50000,
        initial_curriculum_step: int = 0,
        seed: int = 42,
        save_path=None,
        *,
        alpha_min: float = 0.02949,
        omega: float = 0.51,
        gamma: float = 0.99,
        scale_modification_value=(0.8172650252856599, 0.8211253690681617, 0.8257273369742982, 0.8311571820651724),
        t_max: int = 20,
        z_init: float = 4.0,
        f_ag: float = 22.92,
        p_max: float = 4.5,
        # ---- extras of the batched implementation (keyword-only) ----
        num_envs: int = 4096,
        num_populations: int = 1,
        device: int = 0,
        chunk_steps: int = 64,
        threads_per_block: int = 256,
        transfer_mode: str = "reference",
        platform_speed: float = 1.6,
        dynamics: Optional[K.DynamicsParameters] = None,
        max_global_steps: Optional[int] = None,
        envs_per_replica: Optional[int] = None,
        merge_every: int = 1,
        tensorboard: bool = False,
        verbose: bool = True,
        direction: str = "x",
        eval_every: Optional[int] = None,
        eval_episodes: int = 1024,
        eval_two_axis: Optional[K.TwoAxisParameters] = None,
        eval_platforms: Optional[Sequence[Sequence[float]]] = None,
    ) -> None:
        np.random.seed(seed)                                        # PKG/trainer.py:45
        if not double_q_learning_agent:
            double_q_learning_agent = DoubleQLearningAgent(curriculum_steps, device=device)
        self._double_q_learning_agent = double_q_learning_agent
        self._curriculum_steps = self._double_q_learning_agent.curriculum_steps
        self._alpha_min, self._omega, self._gamma = alpha_min, omega, gamma
        self._scale_modification_value = list(scale_modification_value)
        self._successive_successful_episodes = successive_successful_episodes
        self._success_rate = success_rate
        self._alpha = self._alpha_min
        self._exploration_rate = 0.0
        self._z_init, self._t_max, self._f_ag, self._p_max = z_init, t_max, f_ag, p_max
        self._max_num_episodes = max_num_episodes
        self._save_path: Path = Path(save_path) if save_path is not None else ASSETS_PATH / datetime.now().strftime(_TIME_FORMAT)
        self._seed = seed
        self._current_episode = 0
        self._working_curriculum_step = initial_curriculum_step
        self._curriculum_episode_count = 0
        self._successes = deque([], maxlen=successive_successful_episodes)
        # extras
        self._num_envs, self._num_populations, self._device = num_envs, num_populations, device
        self._chunk_steps, self._threads_per_block = chunk_steps, threads_per_block
        self._transfer_mode, self._platform_speed = transfer_mode, platform_speed
        self._dynamics = dynamics or K.DynamicsParameters(z_init=z_init, v_mp=platform_speed)
        self._max_global_steps = max_global_steps
        # one agent with more envs than a CTA should hold -> replica-merge mode (DESIGN.md section 3)
        self._replicas = 1
        if num_populations == 1 and num_envs > 2048:
            if envs_per_replica is None:
                envs_per_replica = replica_shape(num_envs, merge_every)
            self._replicas = -(-num_envs // envs_per_replica)
            self._num_envs = envs_per_replica
            self._threads_per_block = 256 if envs_per_replica >= 256 else (128 if envs_per_replica >= 128 else 32)
        self._merge_every = merge_every
        self._envs_per_agent = self._num_envs * self._replicas      # envs that share one table pair (and one episode budget)
        self._tensorboard, self._verbose = tensorboard, verbose
        if direction not in ("x", "y"):
            raise ValueError("direction must be 'x' or 'y' (training.launch direction:=x|y, training_x.sh / training_y.sh)")
        self._direction = direction
        if eval_every is not None:          # set only when asked for, so a default Trainer pickles exactly as before
            if eval_every < 1 or eval_episodes < 1:
                raise ValueError("eval_every and eval_episodes must be >= 1")
            self._eval_every, self._eval_episodes = eval_every, eval_episodes
        if eval_two_axis is not None:       # likewise stored only when set
            if eval_every is None:
                raise ValueError("eval_two_axis needs eval_every")
            if direction != "x":
                raise ValueError("eval_two_axis flies the x agent on both axes: it needs direction='x'")
            if self._dynamics.accel_mode != "exact" or self._dynamics.dynamics_model != "first_order":
                raise ValueError("eval_two_axis runs the first-order model with the exact acceleration only")
            self._eval_two_axis = eval_two_axis
        if eval_platforms is not None:      # likewise stored only when set
            if eval_every is None:
                raise ValueError("eval_platforms needs eval_every")
            self._eval_platforms = [(float(r), float(v)) for r, v in K.platform_motions(eval_platforms)]
        self._engine = None
        self.history = []             # one dict per chunk (population 0)

    # ------------------------------------------------------------------------------------------------
    # schedules, same formulas and side effects as the reference
    def alpha(self, current_state_action: StateAction):
        """Current learning rate (PKG/trainer.py:88-110)."""
        counter = self._double_q_learning_agent.counter(current_state_action)
        self._alpha = K.alpha_value(counter, self._alpha_min, self._omega)
        if math.isnan(self._alpha):
            raise ValueError(f"Leaning rate cannot be NaN, {counter}, {self._omega}, {self._alpha_min}")
        return self._alpha

    def exploration_rate(self, current_episode: int, current_curriculum_step: int):
        """Current exploration rate (PKG/trainer.py:112-126)."""
        self._exploration_rate = K.exploration_rate(current_episode, current_curriculum_step)
        return self._exploration_rate

    def transfer_learning_ratio(self, curriculum_step: int) -> float:
        """PKG/trainer.py:128-138."""
        return K.transfer_learning_ratio(curriculum_step, self._scale_modification_value)

    # ------------------------------------------------------------------------------------------------
    def __getstate__(self):
        d = dict(self.__dict__)
        d["_engine"] = None
        agent = d.pop("_double_q_learning_agent")
        d["_agent_tables"] = (np.array(agent.Q_table_a), np.array(agent.Q_table_b), np.array(agent.state_action_counter))
        return d

    def __setstate__(self, d):
        tables = d.pop("_agent_tables")
        self.__dict__.update(d)
        agent = DoubleQLearningAgent(len(tables[0]), device=self._device)
        agent.Q_table_a, agent.Q_table_b, agent.state_action_counter = tables
        self._double_q_learning_agent = agent

    def save(self) -> None:
        """Pickle + the three .npy files in the run dir AND its parent (PKG/trainer.py:140-152)."""
        self._save_path.mkdir(parents=True, exist_ok=True)
        with open(self._save_path / "trainer.pickle", "wb") as f:
            pickle.dump(self, f)
        self._double_q_learning_agent.save(self._save_path)
        self._double_q_learning_agent.save(self._save_path / "..")

    @staticmethod
    def load(assets_path: Path = ASSETS_PATH) -> "Trainer":
        """Latest run under ASSETS_PATH (PKG/trainer.py:154-167; the reference's glob/file-name typos are not reproduced)."""
        runs = []
        for p in Path(assets_path).iterdir():
            try:
                runs.append((datetime.strptime(p.name, _TIME_FORMAT), p))
            except ValueError:
                continue
        if not runs:
            raise FileNotFoundError(f"no run directory under {assets_path}")
        save_path = max(runs)[1]
        with open(save_path / "trainer.pickle", "rb") as f:
            trainer = pickle.load(f)
        trainer._double_q_learning_agent = DoubleQLearningAgent.load(save_path)
        return trainer

    # ------------------------------------------------------------------------------------------------
    def _make_engine(self):
        from .engine import Engine
        tp = K.TrainerParameters(
            curriculum_steps=self._curriculum_steps, successive_successful_episodes=self._successive_successful_episodes,
            success_rate=self._success_rate, max_num_episodes=self._max_num_episodes * self._envs_per_agent, alpha_min=self._alpha_min,
            omega=self._omega, gamma=self._gamma, scale_modification_value=self._scale_modification_value,
            transfer_mode=self._transfer_mode)
        mp = K.MdpParameters(f_ag=self._f_ag, t_max=self._t_max, p_max=self._p_max)
        P, R = self._num_populations, self._replicas
        if R > 1:
            eng = Engine(R, self._num_envs, device=self._device, threads_per_block=self._threads_per_block,
                         seeds=[self._seed] * R, population_ids=list(range(R)), v_mp=[self._platform_speed] * R,
                         replicas_per_population=R, axes=[self._direction] * R, mp=mp, dp=self._dynamics, tp=tp)
            P = R
        else:
            eng = Engine(P, self._num_envs, device=self._device, threads_per_block=self._threads_per_block,
                         seeds=[self._seed + p for p in range(P)], population_ids=list(range(P)),
                         v_mp=[self._platform_speed] * P, axes=[self._direction] * P, mp=mp, dp=self._dynamics, tp=tp)
        agent = self._double_q_learning_agent
        for p in range(P):
            eng.set_tables(p, agent.Q_table_a, agent.Q_table_b, agent.state_action_counter)
        return eng

    def _sync_agent_from_device(self, population: int = 0):
        qa, qb, cnt = self._engine.get_tables(population)
        agent = self._double_q_learning_agent
        agent.Q_table_a, agent.Q_table_b, agent.state_action_counter = qa, qb, cnt

    def curriculum_training(self):
        """PKG/trainer.py:169-245, batched: all envs of all populations advance `chunk_steps` global steps per launch."""
        self._engine = eng = self._make_engine()
        eng.reset(self._working_curriculum_step)
        info: Dict[str, Any] = {}
        prev = eng.population_state()
        global_steps = chunks = 0
        while True:
            if self._replicas > 1:
                eng.train_merged(self._chunk_steps, self._merge_every)
            else:
                eng.train(self._chunk_steps)
            eng.check_errors()
            global_steps += self._chunk_steps
            chunks += 1
            ps = eng.population_state()
            p0 = ps[0]
            self._working_curriculum_step = int(p0["working_step"])
            pooled_episodes = int(ps["episodes_in_step"].sum()) if self._replicas > 1 else int(p0["episodes_in_step"])
            self._current_episode = pooled_episodes // self._envs_per_agent      # mean per-env episode index in this curriculum step
            self._curriculum_episode_count = int(ps["total_episodes"].sum()) if self._replicas > 1 else int(p0["total_episodes"])
            window = list(p0["window"][: int(p0["window_count"])])
            self._successes = deque(window, maxlen=self._successive_successful_episodes)
            d_ep = int(p0["total_episodes"] - prev[0]["total_episodes"])
            info = {
                "Termination condition": K.TERMINATION_STRINGS.get(int(p0["last_code"]), ""),
                "Number of steps": int(p0["last_steps"]),
                "Cumulative reward": float(p0["last_cumulative"]),
                "Mean reward": float(p0["last_cumulative"]) / max(int(p0["last_steps"]), 1),
                "Curent episode": self._current_episode,
                "Remaining episodes": self._max_num_episodes - self._current_episode + 1,
                "Exploration rate": self.exploration_rate(self._current_episode, self._working_curriculum_step),
                "Learning rate": self._alpha,
                "Success rate": (int(ps["window_sum"].sum()) / (self._successive_successful_episodes * self._replicas)
                                 if self._replicas > 1 else int(p0["window_sum"]) / self._successive_successful_episodes),
                "Global steps": int(p0["t"]), "Env steps": int(ps["total_steps"].sum()), "Episodes in chunk": d_ep,
                "Pooled episodes": pooled_episodes,
            }
            entry = {}
            if self._eval_every is not None and chunks % self._eval_every == 0:
                rates = eng.eval_agents(self._eval_episodes)["success_rate"]      # greedy policies at the live working steps
                info["Greedy success rate"] = float(rates[0])
                entry["Greedy success rates"] = [float(r) for r in rates]
                if self._eval_two_axis is not None:      # every agent on both axes: its policy on x, the mirror image on y
                    rates2 = eng.eval_pairs(self._eval_episodes, [(g, g) for g in range(len(rates))],
                                            two_axis=self._eval_two_axis)["success_rate"]
                    info["Greedy two-axis success rate"] = float(rates2[0])
                    entry["Greedy two-axis success rates"] = [float(r) for r in rates2]
                if self._eval_platforms is not None:     # every agent under each listed platform motion, one launch
                    by_platform = eng.eval_platforms(self._eval_episodes, self._eval_platforms)["success_rate"]
                    info["Greedy success rate by platform"] = [float(r) for r in by_platform[0]]
                    entry["Greedy success rates by platform"] = [[float(r) for r in row] for row in by_platform]
            self.history.append(dict(info, working_step=self._working_curriculum_step, **entry))
            if len(self.history) > 2048:          # bounded: the history is pickled with every checkpoint
                del self.history[:1024]
            advanced = any(int(ps[p]["working_step"]) != int(prev[p]["working_step"]) or int(ps[p]["finished"]) != int(prev[p]["finished"])
                           for p in range(len(ps)))
            if advanced:                       # checkpoint on promotion instead of after every episode
                self._sync_agent_from_device()
                self.save()
            if self._verbose and (advanced or len(self.history) % 50 == 1):
                self.log(info)
            prev = ps
            if all(int(x["finished"]) for x in ps):
                break
            if self._max_global_steps is not None and global_steps >= self._max_global_steps:
                break
        self._sync_agent_from_device()
        self.save()
        return info

    # ------------------------------------------------------------------------------------------------
    def log(self, info: Dict[str, Any], clean=False):
        """PKG/trainer.py:247-303: same scalar tags and console layout, one writer (not one per episode)."""
        if self._tensorboard:
            from torch.utils.tensorboard.writer import SummaryWriter
            writer = SummaryWriter(log_dir=self._save_path / "logs")
            step = self._curriculum_episode_count
            writer.add_scalar("Episode/Success Rate", info["Success rate"], step)
            writer.add_scalar("Episode/Cumulative Reward", info["Cumulative reward"], step)
            writer.add_scalar("Episode/Exploration Rate", info["Exploration rate"], step)
            writer.add_scalar("Episode/Learning Rate", info["Learning rate"], step)
            writer.add_scalar("Episode/Mean reward", info["Mean reward"], step)
            if "Greedy success rate" in info:
                writer.add_scalar("Episode/Greedy Success Rate", info["Greedy success rate"], step)
            if "Greedy two-axis success rate" in info:
                writer.add_scalar("Episode/Greedy Two-Axis Success Rate", info["Greedy two-axis success rate"], step)
            if "Greedy success rate by platform" in info:
                for (r, v), rate in zip(self._eval_platforms, info["Greedy success rate by platform"]):
                    writer.add_scalar(f"Episode/Greedy Success Rate (r={r:g}, v={v:g})", rate, step)
            writer.add_text("Episode/Termination Condition", info["Termination condition"], step)
            writer.close()
        if clean:
            print("\x1b[0;0f", end="")
            print("\x1b[J", end="")
        else:
            print("=" * 80)
        print(f"Curiculum step: {self._working_curriculum_step + 1}")
        print(f"Current episode: {self._current_episode}")
        shown = dict(info)
        shown["Termination condition"] = shown["Termination condition"].replace("SUCCESS", "\x1b[1;32mSUCCESS\x1b[0m")
        shown["Termination condition"] = shown["Termination condition"].replace("FAILURE", "\x1b[1;31mFAILURE\x1b[0m")
        for k, v in shown.items():
            print(f"{k}: {v}")
        print("Press Ctrl-C to exit...")
        if clean:
            print("\x1b[0;0f", end="")
            print("\x1b[J", end="")
            print("\x1b[0m", end="")
        else:
            print("=" * 80)
