"""Starts a simulation -- the counterpart of the reference's scripts/simulation.py (simulation.sh): loads the committed
agents, runs greedy episodes.  Default: ten episodes through the gym surface exactly like the reference's loop
(agent.predict -> env.step, one env); --episodes N > 10 evaluates N episodes on the device in one launch.

    python scripts/simulation.py
    python scripts/simulation.py --episodes 1048576 --two-axis
    python scripts/simulation.py --episodes 4096 --platforms 2:0.4 2:0.8 2:1.2 2:1.6     # landing rate per platform (r_mp:v_mp)
"""
import argparse
import pathlib
import sys

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parent.parent))

from dql_multirotor_landing_b200 import constants as K                                  # noqa: E402
from dql_multirotor_landing_b200.double_q_learning import DoubleQLearningAgent          # noqa: E402
from dql_multirotor_landing_b200.engine import Engine, greedy_policy, mirrored_policy   # noqa: E402
from dql_multirotor_landing_b200.landing_simulation_env import make                     # noqa: E402


def platform_arg(text):
    """R:V -> (r_mp, v_mp)"""
    try:
        r, v = text.split(":")
        return float(r), float(v)
    except ValueError:
        raise argparse.ArgumentTypeError(f"expected R:V (platform amplitude r_mp and speed v_mp), got {text!r}") from None


def log(info, clean=False):
    """scripts/simulation.py:24-47 of the reference."""
    if clean:
        print("\x1b[0;0f\x1b[J", end="")
    else:
        print("=" * 80)
    info = dict(info)
    info["Termination condition"] = (info["Termination condition"].replace("SUCCESS", "\x1b[1;32mSUCCESS\x1b[0m")
                                     .replace("FAILURE", "\x1b[1;31mFAILURE\x1b[0m"))
    for k, v in info.items():
        print(f"{k}: {v}")
    print("Press Ctrl-C to exit...")
    if not clean:
        print("=" * 80)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--episodes", type=int, default=10)
    ap.add_argument("--two-axis", action="store_true", help="both agents act (the reference leaves the y action disabled)")
    ap.add_argument("--assets", default=None, help="directory with Q_table_a.npy / Q_table_b.npy / state_action_count.npy")
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--platforms", type=platform_arg, nargs="+", default=None, metavar="R:V",
                    help="greedy landing rate of the agent under each platform motion (amplitude r_mp, speed v_mp), one launch")
    a = ap.parse_args()
    agent_x = DoubleQLearningAgent.load(a.assets) if a.assets else DoubleQLearningAgent.load()
    agent_y = DoubleQLearningAgent.load(a.assets) if a.assets else DoubleQLearningAgent.load()
    if a.platforms:
        K.platform_motions(a.platforms)          # ValueError for a malformed list, before the device is touched
        eng = Engine(1, 1, seeds=[a.seed])
        eng.set_tables(0, agent_x.Q_table_a, agent_x.Q_table_b, agent_x.state_action_counter)
        res = eng.eval_platforms(a.episodes, a.platforms, working_step=eng.tp.curriculum_steps - 1)
        print(f"episodes per platform: {a.episodes}  (float32 greedy policy of the agent's tables, working step {eng.tp.curriculum_steps - 1})")
        for (r, v), rate, steps in zip(res["platforms"], res["success_rate"][0], res["steps"][0]):
            print(f"  r_mp = {r:g}  v_mp = {v:g}: landed {rate:.4f}  env-steps {steps}")
        eng.close()
    elif a.episodes <= 10 and not a.two_axis:
        env = make("Landing-Simulation-v0", seed=a.seed)
        for current_episode in range(a.episodes):
            current_state_x, current_state_y = env.reset()
            done = False
            while not done:
                action_x = agent_x.predict(current_state_x)
                action_y = agent_y.predict(current_state_y)
                current_state_x, current_state_y, done, info = env.step(action_x, action_y)
            info["current_episode"] = current_episode + 1
            log(info)
        env.close()
    else:
        pol_x = greedy_policy(agent_x.Q_table_a, agent_x.Q_table_b)
        eng = Engine(1, 1, seeds=[a.seed])
        if a.two_axis:
            ta = K.TwoAxisParameters(trajectory=K.TRAJ_RECTILINEAR_XY, y_action_enabled=True, y_init_enabled=True)
            res = eng.eval_greedy_2d(pol_x, mirrored_policy(pol_x), a.episodes, two_axis=ta, seed=a.seed)
        else:
            res = eng.eval_greedy(pol_x, a.episodes)
        hist = res["termination_hist"]
        print(f"episodes: {res['episodes']}  env-steps: {res['steps']}")
        for code, n in enumerate(hist):
            if n:
                print(f"  {K.TERMINATION_STRINGS.get(code, code)}: {n} ({n / res['episodes']:.4f})")
        eng.close()
