#!/usr/bin/env python
"""bench.py — frame-pairs/s and candidate-evals/s of the stereo block-search hot path.

Workload (BASELINE.json configs[1], "C2" in SURVEY.md 8(d)): a batch of 256 synthetic
640x480 grayscale pairs per GPU, dense template sweep — every 16x16 window, stride 1,
full-row search range (x' in [0, x]), SAD cost, first-minimum selection, then the
reference's ResolveMatchList over the winners on the device (resolved disparity map).
290 625 windows and 90 965 625 candidate evaluations per pair.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...     (one rank per GPU; no data-path collective)

`value`  : pairs/s of the whole step (matching kernel + resolve kernel) with the frames already
           resident in HBM (CUDA events on the launching stream, max over ranks).
`e2e`    : pairs/s through the C-ABI streaming ring with HOST (pinned) buffers — H2D of every
           frame and D2H of every result inside the timed region. The record that crosses PCIe
           is named in e2e.outputs; the same step with wider records is reported beside it.
`roofline`: the sliding-window kernel is integer-ALU bound; achieved = candidate evals/s of the
           MATCHING KERNEL ALONE (its own timed loop, CUDA events) x the ALU-pipe lane-ops one
           evaluation needs in this formulation (DESIGN.md), peak = the VABSDIFF4.U8.ACC issue
           rate measured on this GPU in this run.
`configs`: the other BASELINE configurations on the same line (C3 device-resident, C4 this rank's
           shard of the 4096-pair 1080p batch device-resident and end to end, C5 paired
           unsynchronised streams end to end), each with its own parity flag.
`--dump-outputs DIR`: after the timed steps, what the last step computed for rank 0 — resolved_disparity_u16,
           disparity_u16 and raw_cost_u16 of DUMP_PAIRS pairs drawn with a fixed seed, [pairs, rows, cols] —
           as DIR/<name>.npy in float32 (NO_DISPARITY stays 65535). The inputs are seeded, so two builds run
           with the same arguments can be compared output for output.
`cpu_baseline` / `--impl reference`: the CPU arms, timed on the box's host cores on a bounded
           sample of the same workload: `sliding` (oracle/sliding_sad_cpu.c — the GPU kernel's own
           formulation, OpenMP, all cores; this is the arm `--impl reference` reports, so that the
           GPU/CPU ratio reads as hardware, not as algorithm), `direct` (the direct-form oracle
           port) and `opencv` (cv2.matchTemplate TM_SQDIFF, the nearest OpenCV has: it has no SAD
           mode). The reference repo has no pixel path and cannot be built here (MSVC + OpenCV 3.0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, TW, TH = 640, 480, 16, 16
PAIRS_PER_GPU = 256
# ALU-pipe thread-instructions one candidate evaluation needs in the sliding-window formulation
# (DESIGN.md "roofline"): VABSDIFF4.U8.ACC for the row entering the window, one for the row
# leaving it, and one VIMNMX at twice the VABSDIFF4 issue rate (counted 0.5).
ALU_OPS_PER_EVAL = 2.5
HOST_BIN = os.path.join(ROOT, "unsynchronized_stereo_vision_proj325_b200", "usv_host_test")
DUMP_PAIRS = 16  # 3 arrays x 16 pairs x 290 625 windows x 4 B = 56 MB


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (recipe in B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append((time.time(), [c.strip() for c in line.split(",")]))
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()

    def summary(self, t0, t1):
        rows = [r for t, r in self.rows if t0 <= t <= t1 and len(r) >= 9] or [r for _, r in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        for r in rows:
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "power_w_max": max(float(r[3]) for r in rows),
                "samples": len(rows), "reasons": sorted(reasons)}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def expected_row(oracle, left, right, params, r, nx):
    """Oracle answer for window row r of one gray pair: (disparity_u16, raw cost u32, resolved disparity_u16) — the winners of
    the direct-form oracle, then the reference's ResolveMatchList (restated) over the row's accepted records (records of
    different rows never share a RightIndex, so the row is a closed group of the list)."""
    from unsynchronized_stereo_vision_proj325_b200 import _abi
    ri, rc, _ = oracle.match_dense_rows(left, right, params, int(r), int(r) + 1, threads=host_cores())
    has = ri != _abi.NO_MATCH
    xr = ri.astype(np.int64) - r * nx
    d = np.arange(nx) - xr if params.camera_side == _abi.LEFT_CAM else xr - np.arange(nx)
    exp_d = np.where(has, d, 0xFFFF).astype(np.uint16)
    recs = np.zeros(nx, _abi.MATCH_DTYPE)
    recs["LeftIndex"], recs["RightIndex"] = np.arange(nx) + r * nx, ri
    recs["MatchValue"] = rc / (255.0 * params.tmpl_w * params.tmpl_h)
    alive = np.zeros(nx, bool)
    alive[np.unique(oracle.resolve_match_list(recs[has])["LeftIndex"]) - r * nx] = True
    return exp_d, rc, np.where(alive, exp_d, 0xFFFF).astype(np.uint16)


# ------------------------------------------------------------------------------------------------
# CPU arms (rank 0 only). The oracle is the checker and the CPU baseline, never the product.
# ------------------------------------------------------------------------------------------------
def cpu_sample_sliding(params, seconds=10.0, seed=325):
    """oracle/sliding_sad_cpu.c on all host cores: whole pairs of the workload, batch after batch, for about `seconds`."""
    from oracle import oracle
    from unsynchronized_stereo_vision_proj325_b200 import _abi, api, synth
    cores = host_cores()
    n_src = max(8, 2 * cores)  # enough (pair, band) tasks for every core
    left, right = synth.make_pairs(n_src, W, H, 1, shift=37, noise_sigma=2.0, seed=seed)
    f = _abi.frame_desc_for(left)
    nx, ny, ev_pair = api.grid_dims(f, params)
    oracle.match_dense_sliding(left[:2], right[:2], params, threads=cores)  # warm-up / page-in
    pairs, evals, t_used = 0, 0, 0.0
    while t_used < seconds:
        t0 = time.perf_counter()
        _, _, ev = oracle.match_dense_sliding(left, right, params, threads=cores)
        t_used += time.perf_counter() - t0
        evals += ev
        pairs += n_src
    return {"evals": evals, "seconds": t_used, "pairs": pairs, "cores": cores, "evals_per_pair": ev_pair,
            "pairs_per_s": pairs / t_used, "evals_per_s": evals / t_used}


def cpu_sample_direct(params, seconds=6.0, seed=325):
    """The direct-form oracle port (tw*th byte-ops per candidate) on all host cores: whole window rows for about `seconds`."""
    from oracle import oracle
    from unsynchronized_stereo_vision_proj325_b200 import _abi, api, synth
    n_src = 4
    left, right = synth.make_pairs(n_src, W, H, 1, shift=37, noise_sigma=2.0, seed=seed)
    f = _abi.frame_desc_for(left)
    nx, ny, ev_pair = api.grid_dims(f, params)
    cores = host_cores()
    oracle.match_dense_rows(left[0], right[0], params, 0, min(ny, cores), threads=cores)
    rows_done, evals, t_used = 0, 0, 0.0
    chunk = min(ny, 8 * cores)
    while t_used < seconds:
        pair, r0 = (rows_done // ny) % n_src, rows_done % ny
        n = min(chunk, ny - r0)
        t0 = time.perf_counter()
        _, _, ev = oracle.match_dense_rows(left[pair], right[pair], params, r0, r0 + n, threads=cores)
        t_used += time.perf_counter() - t0
        evals += ev
        rows_done += n
    return {"evals": evals, "seconds": t_used, "rows": rows_done, "ny": ny, "cores": cores, "pairs_per_s": evals / ev_pair / t_used,
            "evals_per_s": evals / t_used}


def cpu_sample_opencv(seconds=3.0, seed=325):
    """cv2.matchTemplate(TM_SQDIFF) of 16x16 templates against the whole right frame, one thread: OpenCV's own block matcher
    (it has no SAD mode and no row-restricted search; a candidate evaluation is one template position)."""
    try:
        import cv2
    except Exception as e:
        return {"unavailable": str(e)}
    from unsynchronized_stereo_vision_proj325_b200 import synth
    cv2.setNumThreads(1)
    left, right = synth.make_pairs(1, W, H, 1, shift=37, noise_sigma=2.0, seed=seed)
    L, R = np.ascontiguousarray(left[0]), np.ascontiguousarray(right[0])
    cv2.matchTemplate(R, np.ascontiguousarray(L[0:TH, 0:TW]), cv2.TM_SQDIFF)
    n, t_used, k = 0, 0.0, 0
    while t_used < seconds:
        x, y = (37 * k) % (W - TW), (53 * k) % (H - TH)
        t0 = time.perf_counter()
        res = cv2.matchTemplate(R, np.ascontiguousarray(L[y:y + TH, x:x + TW]), cv2.TM_SQDIFF)
        t_used += time.perf_counter() - t0
        n += res.size
        k += 1
    return {"cand_evals_per_s": n / t_used, "cores": 1, "version": cv2.__version__, "templates": k,
            "what": "cv2.matchTemplate TM_SQDIFF (float32), one 16x16 template against the whole 640x480 frame per call"}


def run_reference(args, rank, world):
    """`--impl reference`: the CPU arm (sliding-window formulation, all host cores). Rank 0 alone works; other ranks exit 0."""
    if rank != 0:
        return
    from unsynchronized_stereo_vision_proj325_b200 import _abi
    params = _abi.make_params(tmpl_w=TW, tmpl_h=TH, cost="sad", distance_kind=_abi.DIST_PINHOLE)
    per_step = max(1.0, min(12.0, 100.0 / max(1, args.steps + args.warmup)))
    for _ in range(args.warmup):
        cpu_sample_sliding(params, seconds=per_step)
    t, ev, pairs, last = 0.0, 0, 0, None
    for _ in range(args.steps):
        last = cpu_sample_sliding(params, seconds=per_step)
        t += last["seconds"]
        ev += last["evals"]
        pairs += last["pairs"]
    pairs_s = ev / last["evals_per_pair"] / t
    sample = "%.1f whole pairs of the same 640x480 workload per step (%.1f s of CPU work per step)" % (pairs / args.steps, per_step)
    direct = cpu_sample_direct(params, seconds=4.0)
    line = {
        "impl": "reference", "metric": "frame-pairs/sec", "value": pairs_s, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cand_evals_per_s": ev / t,
        "cpu_baseline": {"value": pairs_s, "unit": "pairs/s", "cores": last["cores"], "kind": "port", "sample": sample,
                         "arm": "oracle/sliding_sad_cpu.c: the GPU kernel's formulation (column sums slid down the rows, window sums along x), gcc -O3 -march=native, OpenMP",
                         "direct_form": {"value": direct["pairs_per_s"], "unit": "pairs/s", "cand_evals_per_s": direct["evals_per_s"], "cores": direct["cores"]}},
        "e2e": {"value": pairs_s, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference repo has no pixel-level search and is MSVC/OpenCV-3.0 only (unbuildable here): the CPU arm is this repo's "
                "sliding-window CPU implementation of the same search (bit-exact with the direct-form oracle, reference loop order and tie rule)",
    }
    print(json.dumps(line), flush=True)


def workload_config(n_gpus):
    return {"workload": "C2: %d synthetic 640x480 gray pairs per GPU, 16x16 SAD templates, stride 1, full-row range "
                        "(290625 windows, 90965625 candidate evals per pair), first-min + ResolveMatchList on the device" % PAIRS_PER_GPU,
            "pairs_per_gpu": PAIRS_PER_GPU, "global_pairs": PAIRS_PER_GPU * n_gpus, "parallelism": "pairs sharded, no collective",
            "outputs": "resolved_disparity_u16 per window (2 B): the disparity of every match that survives ResolveMatchList; distance = 640-entry table[disparity]",
            "l2": "inputs (157 MB) + outputs (149 MB) + winners scratch (595 MB) per step exceed the 126 MB L2; no explicit flush"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=PAIRS_PER_GPU, help="pairs per GPU (dev only; the contract value is 256)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C3 / C4 / C5 block (dev only)")
    ap.add_argument("--c4-pairs", type=int, default=4096, help="global C4 batch (dev only; BASELINE says 4096)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from unsynchronized_stereo_vision_proj325_b200 import _abi, api, pipeline, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # torch.distributed is measurement plumbing only (barrier + max over ranks); the data path has no collective
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ranks_true(flag):
        if world == 1:
            return bool(flag)
        t = torch.tensor([1.0 if flag else 0.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item() > 0.5)

    n = args.pairs
    params = _abi.make_params(tmpl_w=TW, tmpl_h=TH, cost="sad", distance_kind=_abi.DIST_PINHOLE)
    ctx = api.Context(local_rank)
    left, right = synth.make_pairs(n, W, H, 1, shift=37, noise_sigma=2.0, seed=325 + rank)
    frame = _abi.FrameDesc(W, H, 1, W, W * H)
    nx, ny, ev_pair = api.grid_dims(frame, params)
    n_win = nx * ny
    stream = torch.cuda.current_stream().cuda_stream

    # ---------------- value: inputs resident in HBM, CUDA events on the launching stream -----------
    d_left = torch.from_numpy(np.ascontiguousarray(left)).cuda()
    d_right = torch.from_numpy(np.ascontiguousarray(right)).cuda()
    o_res = torch.empty(n * n_win, dtype=torch.int16, device="cuda")
    o_disp = torch.empty(n * n_win, dtype=torch.int16, device="cuda")
    o_cost = torch.empty(n * n_win, dtype=torch.int16, device="cuda")
    out_step = _abi.Outputs()      # the contract step: generate -> resolve on the device
    out_step.resolved_disparity_u16, out_step.disparity_u16, out_step.raw_cost_u16 = o_res.data_ptr(), o_disp.data_ptr(), o_cost.data_ptr()
    out_kernel = _abi.Outputs()    # the matching kernel alone (the roofline's launch)
    out_kernel.disparity_u16, out_kernel.raw_cost_u16 = o_disp.data_ptr(), o_cost.data_ptr()

    def step_device():
        ctx.match_dense_device(d_left.data_ptr(), d_right.data_ptr(), frame, n, params, out_step, stream)

    def step_kernel_only():
        ctx.match_dense_device(d_left.data_ptr(), d_right.data_ptr(), frame, n, params, out_kernel, stream)

    def timed_loop(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step_device()
    launches0 = ctx.launch_count
    t_clk0 = time.time()
    ms_total = timed_loop(step_device, args.steps)
    launches = ctx.launch_count - launches0
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        pairs = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_PAIRS), replace=False))
        for name, o in (("resolved_disparity_u16", o_res), ("disparity_u16", o_disp), ("raw_cost_u16", o_cost)):
            a = np.stack([o[int(i) * n_win:(int(i) + 1) * n_win].cpu().numpy().view(np.uint16) for i in pairs])
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a.astype(np.float32).reshape(len(pairs), ny, nx))
    ms_step = ms_total / args.steps
    value = world * n * args.steps / (ms_total * 1e-3)
    # the matching kernel alone, same inputs: the roofline's launch
    for _ in range(2):
        step_kernel_only()
    ms_kernel = timed_loop(step_kernel_only, args.steps) / args.steps
    kernel_name = ctx.last_kernel
    kernel_pairs_s = n / (ms_kernel * 1e-3)      # per GPU
    evals_s = value * ev_pair

    # parity of the timed launches' output against the oracle (rank 0): 8 window rows spread over 4 pairs — winners' cost and
    # disparity, and the resolved map against the reference's ResolveMatchList (restated) over that row's winners
    parity = None
    if rank == 0:
        try:
            from oracle import oracle
            ok, checked = True, []
            res_h = o_res.view(n, ny, nx)
            for pair, rows in ((0, (0, 232)), (n // 3, (100, ny - 1)), ((2 * n) // 3, (7, 300)), (n - 1, (150, ny - 1))):
                for r in rows:
                    exp_d, exp_c, exp_r = expected_row(oracle, left[pair], right[pair], params, r, nx)
                    base = pair * n_win + r * nx
                    got_c = o_cost[base:base + nx].cpu().numpy().view(np.uint16).astype(np.uint32)
                    got_d = o_disp[base:base + nx].cpu().numpy().view(np.uint16)
                    ok = ok and bool(np.array_equal(got_c, exp_c) and np.array_equal(got_d, exp_d))
                    ok = ok and bool(np.array_equal(res_h[pair, r].cpu().numpy().view(np.uint16), exp_r))
                    checked.append([pair, r])
            parity = {"ok": ok, "rows_checked": checked, "what": "raw cost, disparity and resolved disparity of whole window rows, bit-exact"}
        except Exception as e:  # the oracle is optional at bench time
            parity = {"ok": None, "unchecked": str(e)}

    # ---------------- roofline denominator: live VABSDIFF4 issue rate ---------------------------------
    peak_lane = ctx.probe_issue_rate(0, 25.0)
    achieved_lane = kernel_pairs_s * ev_pair * ALU_OPS_PER_EVAL
    out_bytes_kernel = 4  # disparity_u16 + raw_cost_u16
    algo_bytes = 2 * W * H + out_bytes_kernel * n_win  # per pair, matching kernel
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        hbm_src = "measured"
    except Exception:
        hbm_peak, hbm_src = 6650.0, "fallback"
    traffic, warp_inst_pair = None, None
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "dense_traffic.json")))
        traffic = rec["dram_bytes_per_pair"] * n
        warp_inst_pair = rec.get("warp_instructions_per_pair")  # executed warp-instructions, ncu on the same launch
    except Exception:
        pass

    # ---------------- e2e: C-ABI streaming ring, pinned host buffers, H2D + kernels + D2H ------------
    pps = 32 if n % 32 == 0 else n
    n_slots = n // pps

    def measure_e2e(out_mask, check):
        # up to two batches in flight: the ring has two halves of n_slots slots; with depth 2, step k is submitted into
        # half k & 1 before step k - 1 is waited for, so the copies of one step overlap the kernels of its neighbours
        # (every step's H2D and D2H still run inside the timed region, which ends when the last results are on the host)
        st = ctx.stream(frame, params, pairs_per_slot=pps, n_slots=2 * n_slots, mask=out_mask)
        for s in range(2 * n_slots):  # the capture side writes frames straight into the pinned ring
            a = (s % n_slots) * pps
            st.slots[s]["left"][:] = left[a:a + pps]
            st.slots[s]["right"][:] = right[a:a + pps]

        def run_steps(k_steps, depth):
            for k in range(k_steps):
                for s in range(n_slots):
                    st.submit((k & 1) * n_slots + s)
                if depth == 1:
                    for s in range(n_slots):
                        st.wait((k & 1) * n_slots + s)
                elif k > 0:
                    for s in range(n_slots):
                        st.wait(((k - 1) & 1) * n_slots + s)
            if depth == 2:
                for s in range(n_slots):
                    st.wait(((k_steps - 1) & 1) * n_slots + s)

        # warm-up doubles as calibration of the pipeline depth: one GPU alone gains from two steps in flight, several
        # GPUs behind one host lose when copies in both directions overlap all the time (scripts/pcie_probe.py)
        t_cal = {}
        for depth in (1, 2):
            run_steps(1, depth)
            barrier()
            t0 = time.perf_counter()
            run_steps(max(4, args.warmup), depth)
            torch.cuda.synchronize()
            t_cal[depth] = max_over_ranks(time.perf_counter() - t0)
        depth = 1 if t_cal[1] <= 1.03 * t_cal[2] else 2  # two steps in flight only when clearly faster
        forced = os.environ.get("USV_BENCH_E2E_DEPTH")    # measurement aid: pin the depth for A/B runs
        if forced in ("1", "2"):
            depth = int(forced)
        barrier()
        t0 = time.perf_counter()
        run_steps(args.steps, depth)
        torch.cuda.synchronize()
        t = max_over_ranks(time.perf_counter() - t0)
        barrier()
        ok = None
        if check:  # the ring's results equal the device-resident step's (every rank; rows spread over the batch)
            ok = True
            for s, k in ((0, 0), (n_slots // 2, pps // 2), (n_slots - 1, pps - 1)):
                pair = s * pps + k
                got = st.slots[s]["out"]["resolved_disparity_u16"][k]
                ok = ok and bool(np.array_equal(got, o_res[pair * n_win:(pair + 1) * n_win].cpu().numpy().view(np.uint16)))
            ok = all_ranks_true(ok)
        res = (world * n * args.steps / t, st.h2d_bytes_per_pair * n, st.d2h_bytes_per_pair * n, ok, depth, {k: round(v * 1e3, 2) for k, v in t_cal.items()})
        st.close()
        return res

    M = _abi
    e2e_value, h2d, d2h, e2e_ok, e2e_depth, e2e_cal = measure_e2e(M.OUT_RESOLVED_DISPARITY_U16, True)
    t_clk1 = time.time()  # the clock samples cover both timed regions (device-resident and e2e)
    # the same step with wider records, beside e2e and not instead of it: + the winners' integer cost (lossless Match
    # records on the host), and round 1's 8-byte record (no resolve) for continuity
    c_value, c_h2d, c_d2h, _, _, _ = measure_e2e(M.OUT_RESOLVED_DISPARITY_U16 | M.OUT_RAW_COST_U16, False)
    r1_value, _, r1_d2h, _, _, _ = measure_e2e(M.OUT_DISPARITY_U16 | M.OUT_RAW_COST_U16 | M.OUT_DISTANCE_F32, False)

    clocks = None
    if rank == 0:
        sampler.stop()
        clocks = sampler.summary(t_clk0, t_clk1)

    # ---------------- the other BASELINE configurations (C3, C4, C5), outside the C2 timed regions ----
    configs = None
    if not args.no_configs:
        configs = run_configs_block(args, ctx, rank, world, barrier, max_over_ranks, all_ranks_true)

    # ---------------- the C++ drop-in (rank 0 drives every GPU of the run from one process) -----------
    cpp = None
    barrier()
    # the other ranks wait on the HOST (a key of the rendezvous store): a NCCL barrier would keep a spinning kernel on their
    # GPUs, which the C++ workers are about to use
    store = dist.distributed_c10d._get_default_store() if world > 1 else None
    if rank == 0:
        if os.path.exists(HOST_BIN):
            try:
                r = subprocess.run([HOST_BIN, "--bench", str(n * world), str(world), str(max(3, args.steps // 2)), "2"], capture_output=True, text=True, timeout=600)
                cpp = json.loads(r.stdout.strip().splitlines()[-1])
                cpp["value"], cpp["unit"] = cpp.pop("pairs_per_s"), "pairs/s"
            except Exception as e:
                cpp = {"unavailable": str(e)}
        if store is not None:
            store.set("usv_cpp_dropin_done", "1")
    elif store is not None:
        store.wait(["usv_cpp_dropin_done"])
    barrier()

    # ---------------- CPU baseline (rank 0, N = 1 only) ----------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        c = cpu_sample_sliding(params, seconds=10.0)
        d = cpu_sample_direct(params, seconds=5.0)
        cpu = {"value": c["pairs_per_s"], "unit": "pairs/s", "cores": c["cores"], "kind": "port",
               "cand_evals_per_s": c["evals_per_s"],
               "sample": "%d whole pairs of the same workload, %.1f s" % (c["pairs"], c["seconds"]),
               "arm": "sliding: oracle/sliding_sad_cpu.c, the GPU kernel's formulation on the host cores (OpenMP, -O3 -march=native), bit-exact with the direct form",
               "direct_form": {"value": d["pairs_per_s"], "unit": "pairs/s", "cand_evals_per_s": d["evals_per_s"], "cores": d["cores"],
                               "sample": "%d window rows, %.1f s" % (d["rows"], d["seconds"])},
               "opencv": cpu_sample_opencv(3.0)}

    if rank == 0:
        sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
        line = {
            "metric": "frame-pairs/sec", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(world) if n == PAIRS_PER_GPU else dict(workload_config(world), pairs_per_gpu=n, global_pairs=n * world),
            "cand_evals_per_s": evals_s, "kernel": kernel_name + " + dense_resolve_rows_kernel", "gpu_launches": int(launches), "parity_vs_oracle": parity,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "cand_evals_per_s": e2e_value * ev_pair,
                    "api": "usv_stream_submit/usv_stream_wait, %d slots x %d pairs per step, %d step(s) in flight (calibrated in the warm-up)" % (n_slots, pps, e2e_depth),
                    "outputs": "resolved_disparity_u16 per window (2 B): generate -> accept -> ResolveMatchList on the device, one cudaMemcpyAsync per slot; "
                               "H2D 2 x 307 200 B per pair, D2H 581 250 B per pair",
                    "pcie_ceiling_note": "0.61 MB in + 0.58 MB out per pair: at the 64 GB/s each way this pool's 8-GPU hosts deliver with both directions busy "
                                         "(profiles/r1_pcie_probe_n8.json) the H2D side bounds 8 GPUs at ~104 k pairs/s",
                    "matches_device_path": e2e_ok, "calibration_ms_by_depth": e2e_cal,
                    "with_cost": {"value": c_value, "unit": "pairs/s", "h2d_bytes_per_step": int(c_h2d), "d2h_bytes_per_step": int(c_d2h),
                                  "outputs": "resolved_disparity_u16 + raw_cost_u16 per window (4 B): lossless for Match records + distances on the host"},
                    "round1_record": {"value": r1_value, "unit": "pairs/s", "d2h_bytes_per_step": int(r1_d2h),
                                      "outputs": "disparity_u16 + raw_cost_u16 + distance_f32 per window (8 B), no resolve: the record BENCH_r01 moved"},
                    "cpp_dropin": cpp},
            "roofline": {"bound": "alu", "achieved": achieved_lane / 1e12, "peak": peak_lane / 1e12, "unit": "Tlaneop/s",
                         "frac": achieved_lane / peak_lane, "traffic": traffic,
                         "kernel": kernel_name, "kernel_ms_per_launch": ms_kernel, "kernel_pairs_per_s": kernel_pairs_s,
                         "kernel_cand_evals_per_s": kernel_pairs_s * ev_pair,
                         "alu_ops_per_eval": ALU_OPS_PER_EVAL, "peak_source": "VABSDIFF4.U8.ACC issue rate measured in this run (usv_probe_issue_rate)",
                         "direct_form_byteops_per_s": kernel_pairs_s * ev_pair * TW * TH,
                         # how busy the SM's four issue ports are: executed warp-instructions (ncu count of this launch
                         # shape) per second against 4 per clock and SM at the sampled clock
                         "issue_slots": None if not (warp_inst_pair and clocks and clocks.get("sm_mhz")) else {
                             "achieved_gwarpinst_per_s": kernel_pairs_s * warp_inst_pair / 1e9,
                             "peak_gwarpinst_per_s": sms * 4 * clocks["sm_mhz"] * 1e6 / 1e9,
                             "frac": kernel_pairs_s * warp_inst_pair / (sms * 4 * clocks["sm_mhz"] * 1e6)}},
            "roofline_hbm": {"bound": "hbm", "achieved": kernel_pairs_s * algo_bytes / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": kernel_pairs_s * algo_bytes / 1e9 / hbm_peak, "peak_source": hbm_src,
                             "algorithmic_bytes_per_pair": algo_bytes},
            "configs": configs,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def run_configs_block(args, ctx, rank, world, barrier, max_over_ranks, all_ranks_true):
    """C3, C4, C5 of BASELINE.json, short, each with its own parity flag (sampled windows / pairs against the oracle)."""
    import torch
    from unsynchronized_stereo_vision_proj325_b200 import _abi, api, pipeline, synth
    stream = torch.cuda.current_stream().cuda_stream
    out = {}

    def timed(fn, reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fn()
        barrier()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / reps

    try:
        from oracle import oracle
    except Exception:
        oracle = None

    # ---- C3: 1280x720 colour, 32x32 ZNCC, D = 256; 8 pairs per GPU resident in HBM
    try:
        n3 = 16
        l3, r3 = synth.make_pairs(n3, 1280, 720, 3, shift=60, noise_sigma=3.0, seed=33 + rank)
        p3 = _abi.make_params(tmpl_w=32, tmpl_h=32, cost="zncc", search_max=255)
        f3 = _abi.frame_desc_for(l3)
        nx3, ny3, ev3 = api.grid_dims(f3, p3)
        dl, dr = torch.from_numpy(np.ascontiguousarray(l3)).cuda(), torch.from_numpy(np.ascontiguousarray(r3)).cuda()
        o_ri = torch.empty(n3 * nx3 * ny3, dtype=torch.int32, device="cuda")
        o_sc = torch.empty(n3 * nx3 * ny3, dtype=torch.float64, device="cuda")
        o3 = _abi.Outputs()
        o3.right_index, o3.score = o_ri.data_ptr(), o_sc.data_ptr()
        ms = timed(lambda: ctx.match_dense_device(dl.data_ptr(), dr.data_ptr(), f3, n3, p3, o3, stream), 3)
        ok = None
        if oracle is not None:
            rng = np.random.default_rng(5 + rank)
            tx = np.concatenate([rng.integers(0, nx3, 40), [0, nx3 - 1, 127, 128]]).astype(np.int32)
            ty = np.concatenate([rng.integers(0, ny3, 40), [0, ny3 - 1, 300, 301]]).astype(np.int32)
            exp = oracle.match_templates(l3[n3 - 1:], r3[n3 - 1:], tx, ty, p3, mask=_abi.OUT_RIGHT_INDEX | _abi.OUT_SCORE)
            wi = torch.from_numpy((n3 - 1) * nx3 * ny3 + ty.astype(np.int64) * nx3 + tx).cuda()
            ok = bool(np.array_equal(o_ri[wi].cpu().numpy().view(np.uint32), exp["right_index"][0]) and
                      o_sc[wi].cpu().numpy().tobytes() == exp["score"][0].tobytes())
            ok = all_ranks_true(ok)
        out["C3"] = {"workload": "%d pairs per GPU 1280x720x3, 32x32 ZNCC, D = 256, resident in HBM (860561 windows, %d cand evals per pair)" % (n3, ev3),
                     "value": world * n3 / ms * 1e3, "unit": "pairs/s", "cand_evals_per_s": world * n3 * ev3 / ms * 1e3, "ms_per_launch": ms,
                     "kernel": ctx.last_kernel, "outputs": "right_index + f64 score", "parity_vs_oracle": ok,
                     "parity_what": "44 sampled windows of the last pair: index and f64 score bytes"}
        del dl, dr, o_ri, o_sc
    except Exception as e:
        out["C3"] = {"error": str(e)}

    # ---- C4: the 4096-pair 1920x1080 batch (16x16 SAD, D = 256), pairs sharded over the ranks in contiguous blocks
    try:
        total = args.c4_pairs
        lo, hi = pipeline.shard_range(total, rank, world)
        mine, pool = hi - lo, 32
        l4, r4 = synth.make_pairs(pool, 1920, 1080, 1, shift=101, noise_sigma=2.0, seed=44)
        p4 = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="sad", search_max=255)
        f4 = _abi.FrameDesc(1920, 1080, 1, 1920, 1920 * 1080)
        nx4, ny4, ev4 = api.grid_dims(f4, p4)
        nw4 = nx4 * ny4
        # pair g of the batch is pool[g % 32] (a 17 GB batch of distinct noise frames would take minutes to synthesise);
        # the whole shard is resident in HBM: frames and the resolved map of every pair
        idx = torch.arange(lo, hi, device="cuda") % pool
        dl = torch.from_numpy(np.ascontiguousarray(l4)).cuda()[idx].contiguous()
        dr = torch.from_numpy(np.ascontiguousarray(r4)).cuda()[idx].contiguous()
        o_res = torch.empty(mine * nw4, dtype=torch.int16, device="cuda")
        chunk = 256  # launches of 256 pairs: bounds the winners scratch (8 B per window) at 4.2 GB

        def run_c4():
            for a in range(0, mine, chunk):
                m = min(chunk, mine - a)
                o4 = _abi.Outputs()
                o4.resolved_disparity_u16 = o_res.data_ptr() + 2 * a * nw4
                ctx.match_dense_device(dl.data_ptr() + a * f4.frame_stride, dr.data_ptr() + a * f4.frame_stride, f4, m, p4, o4, stream)

        ms = timed(run_c4, 1)
        ok = None
        if oracle is not None:
            g = mine - 1  # last pair of the shard
            src = (lo + g) % pool
            rng = np.random.default_rng(7)
            rows = sorted(set(rng.integers(0, ny4, 3).tolist() + [0, ny4 - 1]))
            ok = True
            for r in rows:
                _, _, exp_r = expected_row(oracle, l4[src], r4[src], p4, r, nx4)
                got = o_res[g * nw4 + r * nx4: g * nw4 + (r + 1) * nx4].cpu().numpy().view(np.uint16)
                ok = ok and bool(np.array_equal(got, exp_r))
            ok = all_ranks_true(ok)
        c4 = {"workload": "%d pairs 1920x1080 gray, 16x16 SAD, D = 256 (2028825 windows, %d cand evals per pair), %d per rank (contiguous blocks), "
                          "drawn from a pool of %d distinct synthetic pairs; generate -> resolve on the device" % (total, ev4, mine, pool),
              "value": total / ms * 1e3, "unit": "pairs/s", "cand_evals_per_s": total * ev4 / ms * 1e3, "seconds_per_batch": ms * 1e-3,
              "kernel": ctx.last_kernel + " + dense_resolve_rows_kernel", "outputs": "resolved_disparity_u16 (2 B per window)", "parity_vs_oracle": ok,
              "parity_what": "5 whole window rows of the shard's last pair: resolved disparity, bit-exact"}
        del dl, dr, o_res
        torch.cuda.empty_cache()
        # end to end: the shard streamed from the page-locked pool through the pinned ring (gather by index), results into the ring
        pps, ns = 8, 6
        st = ctx.stream(f4, p4, pairs_per_slot=pps, n_slots=ns, mask=_abi.OUT_RESOLVED_DISPARITY_U16)
        ctx.host_register(l4)
        ctx.host_register(r4)
        try:
            idx_h = (np.arange(lo, hi) % pool).astype(np.int32)
            sink = np.zeros(1, np.int64)

            def stream_all():
                pending = []
                for b0 in range(0, mine, pps):
                    slot = (b0 // pps) % ns
                    if len(pending) == ns:
                        s_old, c_old = pending.pop(0)
                        st.wait(s_old)
                        sink[0] += int(st.slots[s_old]["out"]["resolved_disparity_u16"][c_old - 1, ::4099].sum())
                    cnt = min(pps, mine - b0)
                    st.submit_gather(slot, l4, idx_h[b0:b0 + cnt], r4, idx_h[b0:b0 + cnt])
                    pending.append((slot, cnt))
                for s_old, c_old in pending:
                    st.wait(s_old)
                    sink[0] += int(st.slots[s_old]["out"]["resolved_disparity_u16"][c_old - 1, ::4099].sum())

            barrier()
            t0 = time.perf_counter()
            stream_all()
            torch.cuda.synchronize()
            t = max_over_ranks(time.perf_counter() - t0)
            c4["e2e"] = {"value": total / t, "unit": "pairs/s", "seconds_per_batch": t, "h2d_bytes_per_pair": st.h2d_bytes_per_pair,
                         "d2h_bytes_per_pair": st.d2h_bytes_per_pair, "api": "usv_stream_submit_gather/usv_stream_wait, %d slots x %d pairs" % (ns, pps)}
        finally:
            st.close()
            ctx.host_unregister(l4)
            ctx.host_unregister(r4)
        out["C4"] = c4
    except Exception as e:
        out["C4"] = {"error": str(e)}

    # ---- C5: two unsynchronised streams of 10 000 frames, host pairing, streamed matching (D = 128), pairs sharded over the ranks
    try:
        n_frames, pool = 10000, 64
        tl, idl = synth.make_timestamps(n_frames, fps=30.0, jitter_sigma=0.002, phase=0.0, drop_prob=0.01, seed=1)
        tr, idr = synth.make_timestamps(n_frames, fps=30.0, jitter_sigma=0.002, phase=0.011, drop_prob=0.01, seed=2)
        t0 = time.perf_counter()
        li, ri, dt = pipeline.pair_streams(tl, tr, 1.0 / 60.0)
        t_pair = time.perf_counter() - t0
        lo, hi = pipeline.shard_range(len(li), rank, world)
        l5, r5 = synth.make_pairs(pool, W, H, 1, shift=37, noise_sigma=2.0, seed=325)
        r5 = np.ascontiguousarray(np.roll(r5, 5, axis=0))  # pair = (left[a], right[b]), a != b in general
        p5 = _abi.make_params(tmpl_w=16, tmpl_h=16, cost="sad", search_max=127)
        f5 = _abi.FrameDesc(W, H, 1, W, W * H)
        nx5, ny5, ev5 = api.grid_dims(f5, p5)
        fl, fr = (idl[li] % pool).astype(np.int32), (idr[ri] % pool).astype(np.int32)
        pps, ns = 32, 6
        st = ctx.stream(f5, p5, pairs_per_slot=pps, n_slots=ns, mask=_abi.OUT_RESOLVED_DISPARITY_U16)
        ctx.host_register(l5)
        ctx.host_register(r5)
        keep = {}
        try:
            def stream_all(record):
                pending = []

                def drain():
                    s_old, b_old, c_old = pending.pop(0)
                    st.wait(s_old)
                    if record and b_old == lo:
                        keep[b_old] = st.slots[s_old]["out"]["resolved_disparity_u16"][0].copy()
                for b0 in range(lo, hi, pps):
                    slot = ((b0 - lo) // pps) % ns
                    if len(pending) == ns:
                        drain()
                    cnt = min(pps, hi - b0)
                    st.submit_gather(slot, l5, fl[b0:b0 + cnt], r5, fr[b0:b0 + cnt])
                    pending.append((slot, b0, cnt))
                while pending:
                    drain()

            stream_all(False)  # warm-up pass
            barrier()
            t0 = time.perf_counter()
            stream_all(True)
            torch.cuda.synchronize()
            t = max_over_ranks(time.perf_counter() - t0)
        finally:
            st.close()
            ctx.host_unregister(l5)
            ctx.host_unregister(r5)
        ok = None
        if oracle is not None and hi > lo:
            a, b = int(fl[lo]), int(fr[lo])
            ok = True
            for r in range(0, ny5, max(1, ny5 // 6)):
                _, _, exp_r = expected_row(oracle, l5[a], r5[b], p5, r, nx5)
                ok = ok and bool(np.array_equal(keep[lo][r * nx5:(r + 1) * nx5], exp_r))
            ok = all_ranks_true(bool(ok))
        out["C5"] = {"workload": "2 x %d frames 640x480 @30 fps, jitter N(0, 2 ms), phase 11 ms, 1 %% drops; nearest-timestamp pairing on the host; 16x16 SAD, "
                                 "D = 128, generate -> resolve on the device; pairs sharded over the ranks; frames from page-locked stores (pool of %d)" % (n_frames, pool),
                     "pairs": int(len(li)), "pairing_seconds": t_pair, "pairing_pairs_per_s": len(li) / t_pair,
                     "value": len(li) / t, "unit": "pairs/s", "e2e": True, "seconds": t, "cand_evals_per_s": len(li) * ev5 / t,
                     "h2d_bytes_per_pair": 2 * W * H, "d2h_bytes_per_pair": 2 * nx5 * ny5,
                     "api": "usv_pair_nearest + usv_stream_submit_gather/usv_stream_wait, %d slots x %d pairs" % (ns, pps),
                     "outputs": "resolved_disparity_u16 (2 B per window)", "parity_vs_oracle": ok,
                     "parity_what": "7 whole window rows of this rank's first streamed pair: resolved disparity, bit-exact"}
    except Exception as e:
        out["C5"] = {"error": str(e)}
    return out


if __name__ == "__main__":
    main()
