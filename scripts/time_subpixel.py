"""Device time of the sub-pixel pass (usv_refine_subpixel_device) behind the dense sweep: the sweep alone against sweep +
refinement, both device-resident, alternated in one process and timed with CUDA events after a warm-up. C2: 256 pairs of
640x480 gray, 16x16 SAD, full range. C3: 16 pairs of 1280x720 colour, 32x32 ZNCC, D = 256.
Prints one JSON line per geometry (GPU name and power limit included); --out FILE also writes them there."""
import argparse
import json
import subprocess
import sys

import numpy as np

sys.path.insert(0, ".")
import torch  # noqa: E402

from unsynchronized_stereo_vision_proj325_b200 import _abi, api, synth  # noqa: E402

CONFIGS = {
    "C2": dict(n=256, w=640, h=480, c=1, params=dict(tmpl_w=16, tmpl_h=16, cost="sad")),
    "C3": dict(n=16, w=1280, h=720, c=3, params=dict(tmpl_w=32, tmpl_h=32, cost="zncc", search_max=255)),
}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = q.stdout.strip().splitlines()[0].split(", ")
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10, help="alternations of the two arms")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = gpu_info()
    ctx = api.Context(0)
    st = torch.cuda.current_stream().cuda_stream
    lines = []
    for cfg_name, cfg in CONFIGS.items():
        n, w, h, c = cfg["n"], cfg["w"], cfg["h"], cfg["c"]
        p = _abi.make_params(**cfg["params"])
        left, right = synth.make_pairs(n, w, h, c, shift=37, noise_sigma=2.0, seed=325)
        dl = torch.from_numpy(np.ascontiguousarray(left)).cuda()
        dr = torch.from_numpy(np.ascontiguousarray(right)).cuda()
        f = _abi.FrameDesc(w, h, c, w * c, w * c * h)
        nx, ny, _ = api.grid_dims(f, p)
        nw = n * nx * ny
        ri = torch.empty(nw, dtype=torch.int32, device="cuda")
        x16 = torch.empty(nw, dtype=torch.int32, device="cuda")
        dist = torch.empty(nw, dtype=torch.float64, device="cuda")
        out = _abi.Outputs()
        out.right_index = ri.data_ptr()

        def sweep():
            ctx.match_dense_device(dl.data_ptr(), dr.data_ptr(), f, n, p, out, st)

        def refine():
            ctx.refine_subpixel_device(dl.data_ptr(), dr.data_ptr(), f, n, p, ri.data_ptr(), x16.data_ptr(), dist.data_ptr(), st)

        arms = {"sweep": [sweep], "sweep_refine": [sweep, refine], "refine": [refine]}
        for fns in arms.values():  # warm-up of every shape the timed window uses
            for _ in range(2):
                for fn in fns:
                    fn()
        torch.cuda.synchronize()
        kernel = ctx.last_kernel
        times = {k: [] for k in arms}
        for _ in range(a.reps):
            for k, fns in arms.items():
                e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
                e0.record()
                for fn in fns:
                    fn()
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1))
        assert api.lib().usv_device_status(ctx._h) == 0
        med = {k: float(np.median(v)) for k, v in times.items()}
        line = {"config": cfg_name, "gpu": name, "power_limit": power, "pairs": n, "windows": nw, "sweep_kernel": kernel,
                "refine_kernel": "subpixel_refine_kernel", "reps": a.reps,
                "sweep_ms": round(med["sweep"], 4), "sweep_refine_ms": round(med["sweep_refine"], 4),
                "refine_ms": round(med["refine"], 4), "refine_ms_from_difference": round(med["sweep_refine"] - med["sweep"], 4),
                "refine_share_of_step": round(med["refine"] / med["sweep_refine"], 4),
                "refined_fraction": float((x16.cpu().numpy() != _abi.NO_SUBPIXEL).mean()),
                "spread_ms": {k: [round(min(v), 4), round(max(v), 4)] for k, v in times.items()}}
        print(json.dumps(line), flush=True)
        lines.append(line)
    ctx.close()
    if a.out:
        with open(a.out, "w") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
