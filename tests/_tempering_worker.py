"""helper process for test_tempering.py::test_nccl_ladder_two_gpus: one rank (= one GPU) with 2 tempered chains, three rounds
of a cycle followed by swap_temperatures"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    rank, world, idfile = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3]
    import numpy as np
    from instagraal_b200.cuda_lib_gl_single import sampler
    from instagraal_b200.replicas import ReplicaSet, nccl_unique_id
    from instagraal_b200.synth import WORKLOADS, make_level
    p8 = np.array([50.0, 9.6, np.float32(0.53 * (9.6 / 50.0) ** -1.5 * 50.0 ** -3), -1.5, 2.0, 900.0, 4.0e5, 0.02], dtype=np.float32)
    level = make_level(WORKLOADS["toy"])
    first = sampler(*level.sampler_args(), device=rank)
    first.set_param_simu(p8)
    rs = ReplicaSet(first, 2, seeds=np.array([10 * rank + 1, 10 * rank + 2], dtype=np.uint64))
    if rank == 0:
        with open(idfile + ".tmp", "wb") as fh:
            fh.write(nccl_unique_id())
        os.replace(idfile + ".tmp", idfile)
    t0 = time.time()
    while not os.path.exists(idfile):
        assert time.time() - t0 < 120
        time.sleep(0.05)
    rs.init_comm(rank, world, open(idfile, "rb").read())
    rs.bomb(seed0=50 + 10 * rank)
    rs.set_ladder([0.0, 1.0, 10.0, 100.0], swap_seed=5)
    rng = np.random.RandomState(rank)
    ladders = []
    for cycle in range(3):
        frags = np.stack([rng.permutation(level.n_frags) for _ in range(2)]).astype(np.int32)
        rs.run_cycle(frags, 5, cycle=cycle, nuisance=True)
        _tried, _acc, ladder = rs.swap_temperatures()
        ladders.append(ladder.tolist())
    stats = {k: v.tolist() for k, v in rs.swap_stats.items()}
    print("RESULT " + json.dumps(dict(rank=rank, ladders=ladders, stats=stats,
                                      temps=[c.chain_temperature for c in rs.chains])), flush=True)
    rs.free()


if __name__ == "__main__":
    main()
