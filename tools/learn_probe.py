"""Learning-quality probe (development aid; SURVEY.md A.4 behavioural golden): success rate per chunk of training at curriculum
step 0, promotion off; beside it the greedy success rate of the agents' live policies (SimulationMdp, 1,024 episodes per agent,
Engine.eval_agents).  One script for the cases DESIGN.md section 3 quotes:

    python tools/learn_probe.py single               one env / 64 / 1,024 envs per CTA (S1 semantics), 8 seeds each
    python tools/learn_probe.py merge                one agent as R replicas x 128 envs, merge interval 1 / 8 / 64
    python tools/learn_probe.py speed                success-rate plateau vs platform speed (128 replicas, merge every step)
    python tools/learn_probe.py R,n_r,merge_every,total_steps[,v_mp]     any replica-merge shape (R = 0: P = 8 independent CTAs of n_r envs)
"""
import json
import pathlib
import sys

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parent.parent))
import numpy as np
from dql_multirotor_landing_b200 import constants as K
from dql_multirotor_landing_b200.engine import Engine


def run(R, n_r, merge_every, total_steps, v_mp=1.6, chunks=6, n_sub=1):
    tp = K.TrainerParameters(success_rate=2.0, max_num_episodes=10 ** 15)
    if R > 0:      # one agent, R replicas merged every `merge_every` global steps
        eng = Engine(R, n_r, threads_per_block=128, seeds=[42] * R, population_ids=list(range(R)), replicas_per_population=R, v_mp=[v_mp] * R, tp=tp)
        P = R
    else:          # 8 independent agents (seeds 42..49), S1 semantics inside each CTA
        P = 8
        eng = Engine(P, n_r, threads_per_block=32 if n_r <= 32 else 128, seeds=list(range(42, 42 + P)), v_mp=[v_mp] * P, tp=tp,
                     dp=K.DynamicsParameters(n_sub=n_sub))
    eng.reset(0)
    chunk = max(total_steps // chunks, 1)
    done, rows, prev_ep, prev_su, prev_hist = 0, [], 0, 0, np.zeros(9)
    while done < total_steps:
        if R > 0:
            eng.train_merged(chunk, merge_every)
        else:
            eng.train(chunk)
        done += chunk
        ps = eng.population_state()
        ep, su = int(ps["total_episodes"].sum()), int(ps["total_successes"].sum())
        hist = ps["termination_hist"].sum(axis=0).astype(float)
        dh = hist - prev_hist
        greedy = float(eng.eval_agents(1024)["success_rate"].mean())      # greedy policies, SimulationMdp, at the live working step
        rows.append(dict(global_steps=done, episodes_per_env=ep // (P * n_r), success_rate_in_chunk=round((su - prev_su) / max(ep - prev_ep, 1), 3),
                         share_success_flyzone_timeout=[round(x, 3) for x in (dh / max(dh.sum(), 1))[[2, 4, 8]]],
                         greedy_success_rate=round(greedy, 3)))
        prev_ep, prev_su, prev_hist = ep, su, hist
    print(json.dumps(dict(replicas=R, envs_per_cta=n_r, merge_every=merge_every if R > 0 else None, v_mp=v_mp, n_sub=n_sub, curve=rows)), flush=True)
    eng.close()


if __name__ == "__main__":
    for a in sys.argv[1:] or ["single"]:
        if a == "single":
            run(0, 1, 0, 600000); run(0, 64, 0, 300000); run(0, 1024, 0, 300000)
        elif a == "merge":
            for R, m in ((8, 8), (64, 8), (512, 8), (512, 1), (512, 64)):
                run(R, 128, m, 300000)
        elif a == "speed":
            for v in (0.0, 0.4, 0.8, 1.0, 1.2, 1.6):
                run(128, 128, 1, 250000, v_mp=v, chunks=5)
        else:
            x = a.split(",")
            run(int(x[0]), int(x[1]), int(x[2]), int(x[3]), float(x[4]) if len(x) > 4 else 1.6)
