#!/usr/bin/env python
"""What per-environment material costs on the step kernel: the bench workload (4096 tier-1 25x25 f32 cloths from the
recorded reset states, aimed touch_cloth actions, reference order, time-sliced launch) run three ways in one process,
alternated round by round:

    plain      clothb200_step_actions_f32 (the batch's material)
    same       clothb200_step_actions_phys_f32, every row = the batch's material (same bits as plain)
    random     clothb200_step_actions_phys_f32, rows drawn per environment (density, ks x[0.5, 2], damping [0, 5],
               plane_friction [0.3, 1], tear_thresh [1.3, 3], gravity [-12, -7])

Every timed launch starts from the same states with the same actions; CUDA events around each launch.  Prints one JSON
line with substeps/s per arm (total substeps run / event time), the GPU's name and power limit.

    python scripts/physics_bench.py [--n 4096] [--rounds 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as exc:  # noqa: BLE001
        return "unknown (%s)" % exc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--seed", type=int, default=1337)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from gym_cloth_b200 import lib as L
    from gym_cloth_b200.batched import BatchedCloth
    if not torch.cuda.is_available():
        raise SystemExit("physics_bench.py measures the GPU: no CUDA device")
    n = args.n
    g = np.load(os.path.join(ROOT, "tests", "golden", "bench_pool_t1.npz"))
    pick = np.arange(n) % len(g["seeds"])
    P = L.default_params()
    bc = BatchedCloth(P, n, dtype=torch.float32)
    p4 = np.zeros((n, bc.N, 4), np.float32); q4 = np.zeros((n, bc.N, 4), np.float32)
    p4[:, :, :3] = g["pos"][pick]; q4[:, :, :3] = g["prev"][pick]
    pos0 = torch.from_numpy(p4).cuda(); prev0 = torch.from_numpy(q4).cuda()
    cov0 = torch.from_numpy(g["start_coverage"][pick].copy()).cuda()
    rng = np.random.RandomState(args.seed)
    a = rng.uniform(-1, 1, size=(n, 4))
    pt = rng.randint(0, bc.N, size=n)
    a[:, :2] = (g["pos"][pick, pt, :2] - 0.5) * 2                  # touch_cloth: aimed at a mesh point of the state
    actions = torch.from_numpy(a.astype(np.float32)).cuda()
    same = torch.tensor([[getattr(P, k) for k in L.PHYSICS_FIELDS] + [0.0, 0.0]], dtype=torch.float64).repeat(n, 1).cuda()
    rnd = same.clone()
    r = np.random.RandomState(args.seed + 1)
    cols = {"density": P.density * r.uniform(0.5, 2, n), "ks": P.ks * r.uniform(0.5, 2, n), "damping": r.uniform(0, 5, n),
            "plane_friction": r.uniform(0.3, 1, n), "tear_thresh": r.uniform(1.3, 3, n), "gravity": r.uniform(-12, -7, n)}
    for i, k in enumerate(L.PHYSICS_FIELDS):
        rnd[:, i] = torch.from_numpy(cols[k]).cuda()
    arms = {"plain": None, "same": same, "random": rnd}

    def launch(phys):
        bc.pos.copy_(pos0); bc.prev.copy_(prev0); bc.flags.zero_(); bc.prev_coverage.copy_(cov0)
        bc.num_steps.zero_(); bc.num_sim_steps.zero_()
        bc.physics = phys
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        bc.step_actions(actions)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3, int(bc.sim_steps.sum().item()), bc.pos.clone()

    for name, ph in arms.items():                                  # warm-up: modules, attributes, slots
        launch(ph)
    res = {k: {"seconds": [], "substeps": []} for k in arms}
    final = {}
    for _ in range(args.rounds):
        for name, ph in arms.items():
            t, s, pos = launch(ph)
            res[name]["seconds"].append(t); res[name]["substeps"].append(s)
            final[name] = pos
    out = {"workload": "%d tier-1 25x25 f32 cloths (bench pool states), one aimed touch_cloth action per launch, "
                       "reference order, time-sliced; CUDA events around each launch" % n,
           "gpu": gpu_info(), "torch": torch.__version__, "rounds": args.rounds,
           "same_bits_as_plain": bool(torch.equal(final["plain"], final["same"]))}
    import ctypes as C
    for name, phys in (("plain", 0), ("per_env", 1)):
        # the kernel each arm launches, as the runtime reports it (cudaOccupancyMaxActiveBlocksPerMultiprocessor,
        # cudaFuncGetAttributes): f32, reference order, constant rest lengths
        v = [C.c_int(0) for _ in range(4)]
        L.check(L.lib().clothb200_step_kernel_info(C.byref(P), 0, 0, 0, phys, *[C.byref(x) for x in v]), "step_kernel_info")
        out.setdefault("kernel", {})[name] = dict(zip(("ctas_per_sm", "registers", "local_bytes", "smem_bytes"), [x.value for x in v]))
    for name in arms:
        sec, sub = np.array(res[name]["seconds"]), np.array(res[name]["substeps"])
        rate = sub / sec
        out[name] = {"substeps_per_s_median": float(np.median(rate)), "substeps_per_s": rate.tolist(),
                     "seconds": sec.tolist(), "substeps": sub.tolist()}
    base = out["plain"]["substeps_per_s_median"]
    for name in ("same", "random"):
        out[name]["vs_plain"] = out[name]["substeps_per_s_median"] / base
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
