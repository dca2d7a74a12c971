"""Cost of the two exact 3-NN kernels (include/b200gs_train.h): the exhaustive b200gs_knn3 against the Morton-tree
b200gs_knn3_tree, on a uniform cube and on Gaussian blobs with 0.1 % outliers 10^4 x out, over point counts from 1 k to
6 M (the exhaustive kernel up to 1 M only: it is O(P^2)).  Where both run, their outputs are compared bit for bit.

Each (cloud, P) is warmed up, then timed with CUDA events in alternating rounds (exhaustive, tree, exhaustive, ...); every
timed window repeats the call enough times to last about 20 ms, and the median over the rounds is reported.  The card's
name and power limit are read in the same run.  Writes one JSON file (--out) and prints a summary line per row.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "sdp-gs_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from b200gs import rasterizer as rz  # noqa: E402
from b200gs._lib import check, lib  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "knn_cost.json"))
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--sizes", default="1000,3000,10000,30000,100000,300000,1000000,3000000,6000000")
ap.add_argument("--exhaustive-max", type=int, default=1_000_000)
A = ap.parse_args()


def cloud(kind, P, seed=0):
    r = np.random.default_rng(seed)
    if kind == "uniform":
        x = r.uniform(-1.0, 1.0, size=(P, 3))
    else:  # blobs + 0.1 % outliers 10^4 x out
        centres = r.uniform(-1.0, 1.0, size=(64, 3))
        x = centres[r.integers(0, 64, P)] + 0.03 * r.normal(size=(P, 3))
        out = r.choice(P, max(P // 1000, 1), replace=False)
        x[out] = 1.0e4 * r.uniform(-1.0, 1.0, size=(out.size, 3))
    return torch.from_numpy(x.astype(np.float32)).cuda()


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
    except Exception as e:  # the power limit is part of the number: say that it could not be read
        name, power, clock = torch.cuda.get_device_name(0), f"unread ({e})", "unread"
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def main():
    torch.cuda.set_device(0)
    rows = []
    for kind in ("uniform", "blobs_outliers"):
        for P in [int(s) for s in A.sizes.split(",")]:
            xyz = cloud(kind, P)
            dist = torch.empty((P,), device="cuda")
            idx = torch.empty((P, 3), dtype=torch.int32, device="cuda")
            nbytes = int(lib.b200gs_knn3_scratch_bytes(P))
            scratch = torch.empty((nbytes,), dtype=torch.uint8, device="cuda")
            calls = dict(tree=lambda: check(lib.b200gs_knn3_tree(P, xyz.data_ptr(), dist.data_ptr(), idx.data_ptr(), scratch.data_ptr(),
                                                                 nbytes, rz._stream())))
            if P <= A.exhaustive_max:
                calls["exhaustive"] = lambda: check(lib.b200gs_knn3(P, xyz.data_ptr(), dist.data_ptr(), idx.data_ptr(), rz._stream()))
            outs, reps = {}, {}
            for name, f in calls.items():  # warm-up, output, and the repeat count of a ~20 ms window
                f()
                torch.cuda.synchronize()
                outs[name] = (dist.clone(), idx.clone())
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); f(); e1.record(); torch.cuda.synchronize()
                reps[name] = max(1, min(1000, math.ceil(20.0 / max(e0.elapsed_time(e1), 1e-3))))
            same = None
            if len(outs) == 2:
                (da, ia), (db, ib) = outs["tree"], outs["exhaustive"]
                same = bool(torch.equal(da.view(torch.int32), db.view(torch.int32)) and torch.equal(ia, ib))
            times = {n: [] for n in calls}
            for _ in range(A.rounds):
                for name in sorted(calls):  # exhaustive, tree, exhaustive, tree, ...
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(reps[name]):
                        calls[name]()
                    e1.record()
                    torch.cuda.synchronize()
                    times[name].append(e0.elapsed_time(e1) / reps[name])
            row = dict(cloud=kind, P=P, ms={n: statistics.median(t) for n, t in times.items()},
                       rounds_ms={n: t for n, t in times.items()}, reps=reps, bit_identical=same)
            rows.append(row)
            print(json.dumps(dict(cloud=kind, P=P, ms=row["ms"], bit_identical=same)), flush=True)
            del xyz, dist, idx, scratch
            torch.cuda.empty_cache()
    res = dict(card=card(), torch=torch.__version__, method="CUDA events, median of %d alternating rounds after warm-up, ~20 ms windows"
               % A.rounds, clouds=dict(uniform="uniform in [-1,1]^3", blobs_outliers="64 Gaussian blobs (sigma 0.03) in [-1,1]^3, "
                                       "0.1 % of the points uniform in [-1e4,1e4]^3"), rows=rows)
    os.makedirs(os.path.dirname(os.path.abspath(A.out)), exist_ok=True)
    with open(A.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
