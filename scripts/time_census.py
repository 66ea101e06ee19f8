"""Device time of the census cost (USV_COST_CENSUS) against the two costs it sits between, on the C2 geometry: 256 pairs
of 640x480 gray, 16x16 templates, stride 1, full range, frames resident in HBM. Three arms, alternated in one process
and timed with CUDA events after a warm-up, each one usv_match_dense_device call writing right_index and disparity_u16:
  census: the census transform of both cameras + dense_census_argmin_kernel
  sad:    dense_sad_argmin_kernel
  zncc:   the one-plane ZNCC sweep the library picks (dense_corr_umma_kernel)
Prints one JSON line (GPU name and power limit included); --out FILE also writes it there."""
import argparse
import json
import subprocess
import sys

import numpy as np

sys.path.insert(0, ".")
import torch  # noqa: E402

from unsynchronized_stereo_vision_proj325_b200 import _abi, api, synth  # noqa: E402

N, W, H = 256, 640, 480


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = q.stdout.strip().splitlines()[0].split(", ")
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10, help="alternations of the three arms")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = gpu_info()
    ctx = api.Context(0)
    st = torch.cuda.current_stream().cuda_stream
    left, right = synth.make_pairs(N, W, H, 1, shift=37, noise_sigma=2.0, seed=325)
    dl = torch.from_numpy(np.ascontiguousarray(left)).cuda()
    dr = torch.from_numpy(np.ascontiguousarray(right)).cuda()
    f = _abi.FrameDesc(W, H, 1, W, W * H)
    arms, kernels, outs = {}, {}, {}
    for cost in ("census", "sad", "zncc"):
        p = _abi.make_params(tmpl_w=16, tmpl_h=16, cost=cost)
        nx, ny, _ = api.grid_dims(f, p)
        ri = torch.empty(N * nx * ny, dtype=torch.int32, device="cuda")
        disp = torch.empty(N * nx * ny, dtype=torch.int16, device="cuda")
        out = _abi.Outputs()
        out.right_index, out.disparity_u16 = ri.data_ptr(), disp.data_ptr()
        outs[cost] = (ri, disp, out)
        arms[cost] = (lambda p=p, out=out: ctx.match_dense_device(dl.data_ptr(), dr.data_ptr(), f, N, p, out, st))
        for _ in range(2):  # warm-up of every shape the timed window uses
            arms[cost]()
        torch.cuda.synchronize()
        kernels[cost] = ctx.last_kernel
    times = {k: [] for k in arms}
    for _ in range(a.reps):
        for k, fn in arms.items():
            e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1))
    assert api.lib().usv_device_status(ctx._h) == 0
    med = {k: float(np.median(v)) for k, v in times.items()}
    true_d = {k: float((outs[k][1].cpu().numpy().view(np.uint16) == 37).mean()) for k in outs}
    line = {"config": "C2", "gpu": name, "power_limit": power, "pairs": N, "kernels": kernels, "reps": a.reps,
            "median_ms": {k: round(v, 4) for k, v in med.items()},
            "kpairs_per_s": {k: round(N / v, 2) for k, v in med.items()},
            "census_over_sad": round(med["census"] / med["sad"], 3), "census_over_zncc": round(med["census"] / med["zncc"], 3),
            "fraction_at_true_disparity": true_d,
            "spread_ms": {k: [round(min(v), 4), round(max(v), 4)] for k, v in times.items()}}
    print(json.dumps(line), flush=True)
    ctx.close()
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
