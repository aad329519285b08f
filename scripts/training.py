"""Starts a training session -- the counterpart of the reference's scripts/training.py (training.sh / training_x.sh /
training_y.sh -> launch/training.launch): no ROS node, no Gazebo; the batched Trainer drives the CUDA path.

    python scripts/training.py                       # x axis, 4 096 envs on one table pair
    python scripts/training.py --direction y --num-envs 65536 --success-rate 0.8
    python scripts/training.py --eval-every 10       # + greedy success rate of the live policy every 10 chunks
    python scripts/training.py --eval-every 10 --eval-two-axis eight    # + its two-axis landing rate (mirror image on y)
"""
import argparse
import pathlib
import sys

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parent.parent))

from dql_multirotor_landing_b200 import constants as K          # noqa: E402
from dql_multirotor_landing_b200.trainer import Trainer         # noqa: E402

# the platforms of the two-axis evaluation: the reference's (y action and y offset disabled), scripts/simulation.py --two-axis
# and bench.py's "eight" (PKG/moving_platform.py:92-111)
TWO_AXIS = {
    "reference": K.TwoAxisParameters(),
    "xy": K.TwoAxisParameters(trajectory=K.TRAJ_RECTILINEAR_XY, y_action_enabled=True, y_init_enabled=True),
    "eight": K.TwoAxisParameters(trajectory=K.TRAJ_EIGHT, r_x=3.0, v_x=0.8, r_y=3.0, y_action_enabled=True, y_init_enabled=True),
}

if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--direction", choices=["x", "y"], default="x", help="launch/training.launch direction:=x|y")
    ap.add_argument("--num-envs", type=int, default=4096)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--success-rate", type=float, default=0.96, help="promotion threshold (PKG/trainer.py:25)")
    ap.add_argument("--max-global-steps", type=int, default=None)
    ap.add_argument("--save-path", default=None)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--noise", action="store_true", help="manager_node's default observation noise (0.25 m, 0.1 m/s)")
    ap.add_argument("--kalman", action="store_true", help="the observation node's Kalman-filtered acceleration estimate")
    ap.add_argument("--second-order", action="store_true", help="second-order attitude + vertical PID dynamics")
    ap.add_argument("--eval-every", type=int, default=None, metavar="N",
                    help="log the greedy policy's SimulationMdp success rate after every N-th chunk (off by default)")
    ap.add_argument("--eval-two-axis", choices=sorted(TWO_AXIS), default=None,
                    help="with --eval-every: also the two-axis greedy landing rate, the x policy on x and its mirror image on y, "
                         "on this platform (the presets of scripts/simulation.py and bench.py)")
    a = ap.parse_args()
    if a.eval_two_axis and a.eval_every is None:
        ap.error("--eval-two-axis needs --eval-every")
    dp = K.DynamicsParameters(n_sub=4 if (a.kalman or a.second_order) else 1,
                              noise_pos_sd=0.25 if a.noise else 0.0, noise_vel_sd=0.1 if a.noise else 0.0,
                              accel_mode="kalman_reference" if a.kalman else "exact",
                              dynamics_model="second_order" if a.second_order else "first_order")
    trainer = Trainer(seed=a.seed, success_rate=a.success_rate, save_path=a.save_path, num_envs=a.num_envs, device=a.device,
                      direction=a.direction, max_global_steps=a.max_global_steps, dynamics=dp,
                      eval_every=a.eval_every, eval_two_axis=TWO_AXIS[a.eval_two_axis] if a.eval_two_axis else None)
    info = trainer.curriculum_training()
    trainer.log(info, clean=False)
