"""Developer tool (GPU box): what camera gradients cost.  For each shape, one view, two persistent sessions over the same
inputs -- the default backward and RasterSession(camera_grads=True) -- each captured into a CUDA graph of its whole
forward+backward step.  Rounds of graph replays alternate between the two (L2 flushed before every step, as bench.py
does), then eager steps give the per-stage CUDA-event times (b200gs_profile_*).  Prints one JSON line with the GPU's
name and power limit.
    python tools/camera_grad_cost.py [--shapes llff_fern_3view,stress_train] [--rounds 10] [--steps 20]"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "sdp-gs_b200"))
import torch  # noqa: E402

import bench  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--shapes", default="llff_fern_3view,stress_train")
ap.add_argument("--rounds", type=int, default=10)
ap.add_argument("--steps", type=int, default=20)
a = ap.parse_args()
from b200gs import _lib  # noqa: E402
from b200gs import rasterizer as rz  # noqa: E402

dev = torch.device("cuda", 0)
torch.cuda.set_device(0)
flush_buf = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)


def replay_ms(graph, steps):
    """Mean ms per step over `steps` replays, each bracketed by events after an L2 flush."""
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for e0, e1 in evs:
        flush_buf.zero_()
        e0.record()
        graph.replay()
        e1.record()
    torch.cuda.synchronize()
    return sum(e0.elapsed_time(e1) for e0, e1 in evs) / steps


def stage_us(session, steps):
    _lib.lib.b200gs_profile_enable(1)
    for i in range(steps + 2):
        if i == 2:
            _lib.lib.b200gs_profile_read(None, None, 1)
        flush_buf.zero_()
        session.step()
    arr, cnt = (C.c_double * 10)(), (C.c_int64 * 10)()
    _lib.lib.b200gs_profile_read(arr, cnt, 1)
    _lib.lib.b200gs_profile_enable(0)
    return {bench.STAGES[i]: round(1000 * arr[i] / steps, 2) for i in range(10)}


def measure(name):
    wl = bench.Workload(name, "extended", dev, views=1)
    P, cam = wl.scene.P, wl.cams[0]
    rs = wl.settings(cam, P)
    L = rz._forward_impl(rs, wl.devt["means3D"], wl.devt["shs"], None, wl.devt["opacities"], wl.devt["scales"], wl.devt["rotations"],
                         None, None, wl.devt["features"], rs.confidence, True)[0]
    sessions = {}
    for mode in ("default", "camera"):
        s = rz.RasterSession(wl.settings(cam, P), means3D=wl.devt["means3D"], opacities=wl.devt["opacities"], shs=wl.devt["shs"],
                             scales=wl.devt["scales"], rotations=wl.devt["rotations"], language_feature_precomp=wl.devt["features"],
                             extended=True, capacity=int(L * 1.25) + 1024, camera_grads=mode == "camera")
        for k, c in zip(("color", "depth", "alpha", "feature"), wl.cot[0]):
            s.cot[k].copy_(c)
        sessions[mode] = s.capture()
    for s in sessions.values():  # warm-up
        replay_ms(s.graph, 5)
    times = {m: [] for m in sessions}
    for _ in range(a.rounds):
        for m, s in sessions.items():
            times[m].append(replay_ms(s.graph, a.steps))
    stages = {m: stage_us(s, a.steps) for m, s in sessions.items()}
    for s in sessions.values():
        assert s.status()[1] == 0
    cg = sessions["camera"].camera_grads
    assert all(bool(torch.isfinite(t).all()) for t in cg.values())
    med = {m: statistics.median(v) for m, v in times.items()}
    return dict(P=P, W=cam.width, H=cam.height, L=int(L),
                step_us={m: round(1000 * v, 1) for m, v in med.items()},
                step_us_rounds={m: [round(1000 * x, 1) for x in v] for m, v in times.items()},
                camera_over_default=round(med["camera"] / med["default"] - 1.0, 4),
                stages_us=stages)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True).stdout.strip()
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q)


print(json.dumps(dict(tool="camera_grad_cost", gpu=gpu_info(), rounds=a.rounds, steps=a.steps,
                      shapes={n: measure(n) for n in a.shapes.split(",")})))
