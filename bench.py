#!/usr/bin/env python
"""bench.py — RDO candidate blocks/s on the BASELINE.json workload (configs[1]).

Workload "1080p-8bit-speed6-me16x16" (one *step* = one pass of the hot path over one batch):
  a lookahead batch of F 1920x1080 8-bit frame pairs (cur, ref) resident in HBM; for every
  16x16 block (8160 per frame)
    * SAD  over CAND_SAD  full-pel MV candidates (get_fullpel_mv_rd, me.rs:1386) + per-block
      first-min winner (me.rs:898),
    * SATD over CAND_SATD candidates (the sub-pel / mode-pruning distortion, dist.rs:156),
    * forward DCT_DCT 16x16 of the winner's residual (forward_transform, forward.rs:71)
      [added once the transform kernels land; reported in config.legs].
  value = candidate blocks evaluated per second, whole job (all ranks).
  F is sized so that planes + descriptors exceed the 126 MB L2 (config.l2: "inputs>L2").

JSON contract: see the task statement; extra objects `roofline`, `cpu_baseline`, `e2e`,
`clocks`, `gpu_launches`.  `--impl reference` times the CPU oracle (the reference's
algorithm restated in C; rav1e itself cannot be built here: no rustc/nasm) with all host
threads on a bounded sample of the same workload.
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

W, H, PAD = 1920, 1080, 96
BW = BH = 16
CAND_SAD = 64     # full-pel candidates per block and reference (predictors + diamond + UMH head)
CAND_SATD = 8     # sub-pel diamond / mode-pruning SATD candidates per block
MV_RANGE_PX = 64  # candidates uniform in +-64 px (SURVEY §8d cfg 2b)
LAMBDA = 6400
FRAMES_PER_GPU = 32
METRIC = "RDO candidate blocks/s (SAD+SATD+fwd-txfm) 1080p speed-6"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples nvidia-smi clocks/throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            t0 = time.perf_counter()       # nvidia-smi takes a few 100 ms to start: the first sample
            while not self.lines and time.perf_counter() - t0 < 5.0:   # must exist before the load begins
                time.sleep(0.01)
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "samples": len(sm),
                "reasons": sorted(reasons)}


def synth_frame_pair(seed):
    """cur(x,y) = ref(x+dx, y+dy) + noise on a padded canvas (borders carry real pixels)."""
    rng = np.random.default_rng(seed)
    ref = rng.integers(0, 256, (H + 2 * PAD, W + 2 * PAD), dtype=np.uint8)
    dx, dy = int(rng.integers(-8, 9)), int(rng.integers(-8, 9))
    cur = np.roll(ref, (-dy, -dx), axis=(0, 1)).astype(np.int16)
    cur += rng.integers(-2, 3, cur.shape, dtype=np.int16)
    return np.clip(cur, 0, 255).astype(np.uint8), ref


def grid_blocks():
    from rav1e_b200 import backend as B
    xs = np.arange(0, W - BW + 1, BW)
    ys = np.arange(0, H - BH + 1, BH)     # 67 full rows; the 16x8 bottom strip is a different size
    b = np.zeros(len(xs) * len(ys), B.BLOCK_DTYPE)
    b["x"] = np.tile(xs, len(ys))
    b["y"] = np.repeat(ys, len(xs))
    return b


def cand_list(nblocks, per_block, seed):
    from rav1e_b200 import backend as B
    rng = np.random.default_rng(seed)
    n = nblocks * per_block
    c = np.zeros(n, B.CAND_DTYPE)
    c["block"] = np.repeat(np.arange(nblocks, dtype=np.uint32), per_block)
    mv = rng.integers(-MV_RANGE_PX, MV_RANGE_PX + 1, (n, 2), dtype=np.int16) * 8
    c["mv_row"], c["mv_col"] = mv[:, 0], mv[:, 1]
    offs = (np.arange(nblocks + 1, dtype=np.uint64) * per_block).astype(np.uint32)
    return c, offs


# ----------------------------------------------------------------------------- reference arm
def run_reference(args, rank, world):
    if rank != 0:
        return
    from tests import oracle_lib as O
    threads = O.host_threads()
    tiles_mode = args.workload == "4k-tiles"
    blocks = grid_blocks()
    cur_img, ref_img = synth_frame_pair(0)
    ocur, oref = O.Plane(W, H, PAD), O.Plane(W, H, PAD)
    ocur.data[:], oref.data[:] = cur_img, ref_img
    # bounded sample: one 1080p frame pair's worth of 16x16 blocks per step.  The same sample serves the
    # 4K tile workload: its unit is the same 16x16 candidate block (two 960x1088 tiles hold as many
    # blocks as one 1080p frame) and the CPU's cost per block does not depend on the frame size.
    sad_c, _ = cand_list(len(blocks), CAND_SAD, 100)
    satd_c, _ = cand_list(len(blocks), CAND_SATD, 200)
    resid = np.random.default_rng(5).integers(-255, 256, (len(blocks), BH, BW)).astype(np.int16)
    units = len(sad_c) + len(satd_c) + len(resid)

    def step():
        O.fullpel_candidates(ocur, oref, blocks, sad_c, BW, BH, False, LAMBDA, want_cost=True, threads=threads)
        O.fullpel_candidates(ocur, oref, blocks, satd_c, BW, BH, True, LAMBDA, want_cost=True, threads=threads)
        O.forward_transform_batch(resid, 2, 0, 8, threads=threads)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    v = units * args.steps / dt
    sample = (f"1 of {FRAMES_PER_GPU} frame pairs per step: {CAND_SAD} SAD + {CAND_SATD} SATD candidates and "
              f"one 16x16 DCT_DCT per 16x16 block ({units} blocks/step), {threads} threads "
              f"(affinity capped by the cgroup CPU quota)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "blocks/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic",
        "config": {"workload": "4k-8bit-speed6-8tiles (BASELINE configs[4])" if tiles_mode else "1080p-8bit-speed6-me16x16",
                   "sample": sample,
                   "note": "rav1e cannot be built here (no rustc/nasm); this is the C restatement "
                           "of its rust:: kernels (oracle/), OpenMP over candidates"},
        "cpu_baseline": {"value": v, "unit": "blocks/s", "cores": threads, "kind": "port",
                         "sample": sample},
        "e2e": {"value": v, "unit": "blocks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ----------------------------------------------------------------------------- B200 arm
def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from rav1e_b200 import backend as B

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # one side stream shared by torch (events, NCCL ordering) and the backend's launches
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    ctx = B.Context(local_rank, use_torch_stream=True)
    assert ctx.L.b200_ctx_get_stream(ctx.h) == stream.cuda_stream

    F = args.frames
    blocks = grid_blocks()
    nb = len(blocks)
    d_blocks = torch.from_numpy(blocks.view(np.uint8)).cuda()
    # 4 distinct synthetic frame pairs uploaded into F distinct device planes (addresses, not
    # content, are what cache behaviour depends on); candidate lists are distinct per frame.
    uniq = [synth_frame_pair(1000 * rank + i) for i in range(min(4, F))]
    planes = []
    import ctypes as C
    for f in range(F):
        cur_img, ref_img = uniq[f % len(uniq)]
        pr = []
        for img in (cur_img, ref_img):
            p = B.Plane()
            ctx.check(ctx.L.b200_plane_alloc(ctx.h, W + 2 * PAD, H + 2 * PAD, 0, 1, C.byref(p)))
            ctx.check(ctx.L.b200_plane_upload(ctx.h, C.byref(p), img.ctypes.data, img.strides[0]))
            q = B.Plane()
            q.data = p.data + PAD * p.stride + PAD
            q.stride, q.width, q.height, q.pad, q.bpp, q.alloc = p.stride, W, H, PAD, 1, None
            pr.append(q)
        planes.append(pr)
    # Descriptors of all F frame pairs, concatenated pair after pair (b200_me_candidates_multi_dev
    # layout: global block indices, one CSR over all blocks).  P pairs go into one launch.
    P = max(1, min(args.pairs_per_launch, F))
    sad_np, satd_np = [], []
    for f in range(F):
        c, offs = cand_list(nb, CAND_SAD, 7 * f + 1 + 100000 * rank)
        c["block"] += f * nb
        sad_np.append(c)
        c2, offs2 = cand_list(nb, CAND_SATD, 7 * f + 2 + 100000 * rank)
        c2["block"] += f * nb
        satd_np.append(c2)
    n_sad, n_satd = nb * CAND_SAD, nb * CAND_SATD
    d_sad_c = torch.from_numpy(np.concatenate(sad_np).view(np.uint8)).cuda()
    d_satd_c = torch.from_numpy(np.concatenate(satd_np).view(np.uint8)).cuda()
    del sad_np, satd_np
    d_blocks_all = torch.from_numpy(np.tile(blocks, F).view(np.uint8)).cuda()
    d_offs = torch.from_numpy((np.arange(F * nb + 1, dtype=np.uint64) * CAND_SAD).astype(np.uint32).view(np.uint8)).cuda()
    d_offs2 = torch.from_numpy((np.arange(F * nb + 1, dtype=np.uint64) * CAND_SATD).astype(np.uint32).view(np.uint8)).cuda()
    d_sad = torch.empty(F * n_sad * 4, dtype=torch.uint8, device="cuda")
    d_satd = torch.empty(F * n_satd * 4, dtype=torch.uint8, device="cuda")
    d_best = torch.empty(F * nb * 16, dtype=torch.uint8, device="cuda")
    d_best2 = torch.empty(F * nb * 16, dtype=torch.uint8, device="cuda")
    d_coef = torch.empty(F * nb * BW * BH, dtype=torch.int16, device="cuda")
    gathered = torch.empty(world * F * nb * 16, dtype=torch.uint8, device="cuda") if world > 1 else None
    p_sad = B.me_params(BW, BH, W, H, LAMBDA, window_hint_px=MV_RANGE_PX)
    p_satd = B.me_params(BW, BH, W, H, LAMBDA, use_satd=True, window_hint_px=MV_RANGE_PX)
    # launch groups: frames [f0, f1) -> one call of each leg.  Offsets/cands keep global block
    # indices, so a group passes the concatenated arrays from its first block / candidate on with
    # indices rebased by the library's pair table (block_end / cand_end are relative to the group).
    groups = []
    for f0 in range(0, F, P):
        f1 = min(F, f0 + P)
        k = f1 - f0
        pairs_sad = B.PlanePairs([planes[f][0] for f in range(f0, f1)], [planes[f][1] for f in range(f0, f1)],
                                 [(i + 1) * nb for i in range(k)], [(i + 1) * n_sad for i in range(k)])
        pairs_satd = B.PlanePairs([planes[f][0] for f in range(f0, f1)], [planes[f][1] for f in range(f0, f1)],
                                  [(i + 1) * nb for i in range(k)], [(i + 1) * n_satd for i in range(k)])
        groups.append((f0, k, pairs_sad, pairs_satd))
    # per-group descriptor views: candidates of group g carry block indices relative to the group
    if P < F:
        for f in range(F):
            base = (f // P) * P * nb
            if base:
                v = d_sad_c[f * n_sad * 8:(f + 1) * n_sad * 8].view(torch.int32).view(-1, 2)
                v[:, 0] -= base
                v2 = d_satd_c[f * n_satd * 8:(f + 1) * n_satd * 8].view(torch.int32).view(-1, 2)
                v2[:, 0] -= base
    d_offs_g = d_offs[:(P * nb + 1) * 4]        # identical for every group (uniform list lengths)
    d_offs2_g = d_offs2[:(P * nb + 1) * 4]

    def sad_launch(g):
        f0, k, ps, _ = groups[g]
        ctx.me_candidates_multi_dev(ps, d_blocks_all, k * nb, d_sad_c[f0 * n_sad * 8:], k * n_sad, p_sad,
                                    d_offs_g, None, d_sad[f0 * n_sad * 4:], None, d_best[f0 * nb * 16:])

    def satd_launch(g):
        f0, k, _, ps = groups[g]
        ctx.me_candidates_multi_dev(ps, d_blocks_all, k * nb, d_satd_c[f0 * n_satd * 8:], k * n_satd, p_satd,
                                    d_offs2_g, None, d_satd[f0 * n_satd * 4:], None, d_best2[f0 * nb * 16:])

    def txfm_launch(g):
        f0, k, ps, _ = groups[g]
        # fused diff + TX_16X16 DCT_DCT (8-bit -> i16 coefficients) of the SAD winners
        ctx.fwd_txfm_residual_multi_dev(ps, d_blocks_all, k * nb, d_best[f0 * nb * 16:],
                                        d_coef[f0 * nb * BW * BH:], 2, 0, 8)

    NG = len(groups)
    side = torch.cuda.Stream(device=local_rank)
    ev_sad, ev_comm = torch.cuda.Event(), torch.cuda.Event()

    def step():
        for g in range(NG):
            sad_launch(g)
        if world > 1:   # winners to every rank (the entropy-coder owner): on a side stream as soon as the
            ev_sad.record(stream)        # SAD legs are done, under the SATD and transform legs
            with torch.cuda.stream(side):
                side.wait_event(ev_sad)
                dist.all_gather_into_tensor(gathered, d_best)
                ev_comm.record(side)
        for g in range(NG):
            satd_launch(g)
            txfm_launch(g)
        if world > 1:
            stream.wait_event(ev_comm)   # the step ends when the winners have arrived everywhere

    def timed(fn, reps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    clk = ClockSampler(local_rank)
    if rank == 0:
        clk.start()          # sampled from the warm-up on: the same kernels at the same load
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    l0 = ctx.launches
    ms = timed(step, args.steps)
    launches = ctx.launches - l0
    # the last timed step's outputs, copied on the device before the untimed steps below rewrite them
    snapshot = [t.clone() for t in (d_sad, d_satd, d_best, d_best2, d_coef)] if args.dump_outputs and rank == 0 else None
    for _ in range(int(min(2000, max(0, 250.0 / max(ms / args.steps, 1e-3) - args.steps)))):   # ~0.25 s more of the
        step()                                                   # same steps (untimed): clock samples under load
    torch.cuda.synchronize()
    units_per_step = world * F * (n_sad + n_satd + nb)
    value = units_per_step * args.steps / (ms * 1e-3)

    # ---- roofline of the dominant kernel (candidate-list SAD), timed alone on the same stream
    def sad_only():
        for g in range(NG):
            sad_launch(g)

    def satd_only():
        for g in range(NG):
            satd_launch(g)
    sad_only()
    ms_sad = timed(sad_only, args.steps) / (args.steps * NG)      # ms per launch
    satd_only()
    ms_satd = timed(satd_only, args.steps) / (args.steps * NG)

    def txfm_only():
        for g in range(NG):
            txfm_launch(g)
    txfm_only()
    ms_txfm = timed(txfm_only, args.steps) / (args.steps * NG)
    # clocks / throttle reasons over the warm-up, the timed step region and the per-leg timings above
    clocks = clk.stop() if rank == 0 else None
    # ---- extra leg (not part of `value`): the exhaustive grid full_pixel_me falls back to at
    # speed <= 5 (me.rs:822-846): +-192 x +-64 px, step 4 => up to 97 x 33 = 3201 positions/block
    d_fs = torch.empty(nb * 16, dtype=torch.uint8, device="cuda")
    p_fs = B.me_params(BW, BH, W, H, LAMBDA)
    FS_FRAMES = min(F, 4)

    def fs_only():
        for f in range(FS_FRAMES):
            cur, ref = planes[f]
            ctx.me_full_search_dev(cur, ref, d_blocks, nb, p_fs, 192, 64, 4, d_fs)
    fs_only()
    ms_fs = timed(fs_only, max(2, args.steps // 2)) / (max(2, args.steps // 2) * FS_FRAMES)
    # ---- extra leg (not part of `value`): BASELINE configs[3] - 1080p 10-bit speed-2 inter RDO, sub-pel
    # MC + SATD + forward transform FUSED (b200_subpel_rdo_dev): per 16x16 block the 8 vectors of the
    # sub-pel diamond at radius 4 and 2 around a full-pel centre -> put_8tap(REGULAR) -> SATD + cost ->
    # first minimum -> residual -> DCT_DCT 16x16, one launch per frame pair, nothing but source pixels read
    rng4 = np.random.default_rng(77 + rank)
    img10 = [rng4.integers(0, 1024, (H, W)).astype(np.uint16) for _ in range(2)]
    p10 = [ctx.plane_from_host(im, PAD) for im in img10]
    pattern = np.array([(r * s_, c * s_) for s_ in (4, 2) for r, c in ((1, 0), (0, 1), (-1, 0), (0, -1))])
    centre = rng4.integers(-16, 17, (nb, 2)) * 8
    c4 = np.zeros(nb * 8, B.CAND_DTYPE)
    c4["block"] = np.repeat(np.arange(nb, dtype=np.uint32), 8)
    mv4 = (centre[:, None, :] + pattern[None]).reshape(-1, 2)
    c4["mv_row"], c4["mv_col"] = mv4[:, 0], mv4[:, 1]
    d_c4 = torch.from_numpy(c4.view(np.uint8)).cuda()
    d_o4 = torch.from_numpy((np.arange(nb + 1, dtype=np.uint32) * 8).view(np.uint8)).cuda()
    d_b4 = torch.empty(nb * 16, dtype=torch.uint8, device="cuda")
    d_k4 = torch.empty(nb * 256, dtype=torch.int32, device="cuda")
    p_c4 = B.me_params(BW, BH, W, H, LAMBDA, allow_hp=True, use_satd=True, bit_depth=10)

    def cfg4_only():
        ctx.subpel_rdo_dev(p10[0], p10[1], d_blocks, nb, d_c4, nb * 8, d_o4, p_c4, 0, 2, 0, None, None, None, d_b4, d_k4)
    cfg4_only()
    ms_c4 = timed(cfg4_only, max(2, args.steps // 2)) / max(2, args.steps // 2)
    for pl in p10:
        ctx.plane_free(pl)
    w_in_b, h_in_b = 2 * ((W + 7) >> 3), 2 * ((H + 7) >> 3)
    bx, by = blocks["x"].astype(np.int64), blocks["y"].astype(np.int64)
    mvx_min = np.maximum(-(bx // 4) * 32 - (128 + BW * 8), -(1 << 14) + 1)
    mvx_max = np.minimum((w_in_b - bx // 4 - BW // 4) * 32 + 128 + BW * 8, (1 << 14) - 1)
    mvy_min = np.maximum(-(by // 4) * 32 - (128 + BH * 8), -(1 << 14) + 1)
    mvy_max = np.minimum((h_in_b - by // 4 - BH // 4) * 32 + 128 + BH * 8, (1 << 14) - 1)
    tdiv = lambda a, b: np.sign(a) * (np.abs(a) // b)          # Rust `/` truncates toward zero
    nxp = (np.minimum(192, tdiv(mvx_max, 8)) - np.maximum(-192, tdiv(mvx_min, 8))) // 4 + 1
    nyp = (np.minimum(64, tdiv(mvy_max, 8)) - np.maximum(-64, tdiv(mvy_min, 8))) // 4 + 1
    fs_positions = int((nxp * nyp).sum())

    pairs_per_launch = F / NG
    # SURVEY §8d: 260 B/cand + 256 B/block, x the frame pairs one launch covers
    alg_bytes = int((n_sad * (BW * BH + 4) + nb * BW * BH) * pairs_per_launch)
    peak, peak_src = peaks()
    achieved = alg_bytes / (ms_sad * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        with open(tp) as fh:
            traffic = json.load(fh).get("me_cand_group_u8_16x16_dram_bytes_per_frame_pair")
            if traffic is not None:
                traffic = int(traffic * pairs_per_launch)

    out = None
    # ---- e2e: same metric through the host-buffer C ABI (H2D + kernels + D2H per frame), on every rank
    e2e = run_e2e(ctx, blocks, args, world, dist if world > 1 else None)
    # ---- the 4K tile workload (BASELINE configs[4]) on the same ranks: strong scaling, reported beside the
    # headline so that the N = 1, 2, 4, 8 lines of one series carry both (auto mode; --workload 1080p skips it)
    tiles4k = None
    if args.workload == "auto":
        torch.cuda.synchronize()
        tiles4k = run_b200_tiles(args, rank, world, local_rank, embedded=True)
        torch.cuda.set_stream(stream)
    if rank == 0:
        cpu = run_cpu_baseline(blocks)
        out = {
            "metric": METRIC, "value": value, "unit": "blocks/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": "1080p-8bit-speed6-me16x16", "frames_per_gpu": F,
                       "blocks_per_frame": nb, "block": "16x16",
                       "legs": {"sad_candidates_per_block": CAND_SAD,
                                "satd_candidates_per_block": CAND_SATD,
                                "fwd_txfm_per_block": "1 x TX_16X16 DCT_DCT of the SAD winner's residual"},
                       "mv_range_px": MV_RANGE_PX, "lambda": LAMBDA,
                       "frame_pairs_per_launch": pairs_per_launch,
                       "l2": "inputs>L2 (planes %.0f MB + descriptors %.0f MB per GPU)" % (
                           F * 2 * (W + 2 * PAD) * (H + 2 * PAD) / 1e6, F * (n_sad + n_satd) * 8 / 1e6),
                       "parallelism": f"frames sharded over {world} GPU(s); all-gather of winners"
                       if world > 1 else "1 GPU",
                       "per_launch_ms": {"sad_cand": ms_sad, "satd_cand": ms_satd,
                                         "residual+fwd_txfm": ms_txfm},
                       "extra_legs": {"full_search_grid": {
                           "what": "me_full_search (+-192 x +-64 px, step 4) for every 16x16 block of one frame; "
                                   "not part of `value` (speed 6 disables full search)",
                           "positions_per_launch": fs_positions, "launch_ms": ms_fs,
                           "candidates_per_s": fs_positions / (ms_fs * 1e-3)},
                           "config3_subpel_fused_10bit": {
                               "what": "BASELINE configs[3]: 1080p 10-bit, per 16x16 block 8 sub-pel vectors -> put_8tap(REGULAR) "
                                       "-> SATD + cost -> first minimum -> residual -> DCT_DCT 16x16 in ONE kernel "
                                       "(b200_subpel_rdo_dev); not part of `value`",
                               "blocks_per_launch": nb, "candidates_per_launch": nb * 8, "launch_ms": ms_c4,
                               "blocks_per_s": nb / (ms_c4 * 1e-3), "candidates_per_s": nb * 8 / (ms_c4 * 1e-3),
                               "algorithmic_bytes_per_block": 8 * 23 * 23 * 2 + 256 * 2 + 256 * 4 + 16,
                               "algorithmic_GBps": nb * (8 * 23 * 23 * 2 + 256 * 2 + 256 * 4 + 16) / (ms_c4 * 1e-3) / 1e9}}},
            "roofline": {"kernel": "me_cand_group_u8<16,16,SAD> (candidate-list SAD + cost + argmin)",
                         "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "traffic_source": "static: ncu dram__bytes of the same 32-pair launch recorded in "
                                           "profiles/traffic.json (not re-measured in this run)",
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "launch_ms": ms_sad,
                         # what actually binds this kernel (ncu: DRAM traffic is 0.08x the algorithmic bytes):
                         # warp-instruction issue.  Floor per candidate in the cooperative loop: 1 LDS.128
                         # (parameters) + 4 LDS.32 + 2 funnel shifts + 2 VABSDIFF4.ACC + 1 REDUX = 10.
                         "issue_roof": {"floor_warp_instr_per_candidate": 10,
                                        "peak_candidates_per_s": 148 * 4 * 1.965e9 / 10,
                                        "achieved_candidates_per_s": n_sad * pairs_per_launch / (ms_sad * 1e-3),
                                        "frac": n_sad * pairs_per_launch / (ms_sad * 1e-3) / (148 * 4 * 1.965e9 / 10),
                                        "note": "148 SMs x 4 schedulers x 1 warp instruction per clock at 1965 MHz; "
                                                "the measured kernel issues ~29 per candidate, issue slots 68 % busy, L1TEX 73 % "
                                                "(ncu, profiles/prof_r2l_sad_raw.csv, NOTES_r2.md)"}},
            "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks, "gpu_launches": int(launches),
        }
        if tiles4k is not None:
            out["strong_scaling_4k_tiles"] = tiles4k
        if snapshot is not None:
            s_sad, s_satd, s_best, s_best2, s_coef = (t.cpu().numpy() for t in snapshot)
            winners = lambda b: np.stack([b["cost"], b["sad"], b["mv_row"], b["mv_col"]], axis=1)
            dump_outputs(args.dump_outputs, {
                "sad_candidates": s_sad.view(np.uint32), "satd_candidates": s_satd.view(np.uint32),
                "sad_winners": winners(s_best.view(B.ME_RESULT_DTYPE)),
                "satd_winners": winners(s_best2.view(B.ME_RESULT_DTYPE)),
                "coefficients": s_coef.reshape(F * nb, BW * BH)})
        print(json.dumps(out))
    finish(world, dist)


DUMP_VALUES = 1 << 20      # values kept per output by --dump-outputs (8 MB as float64)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: every output as out_dir/<name>.npy in float64, which holds all of their values exactly.  Rows
    are the step's blocks or candidates, frame after frame.  An output of more than DUMP_VALUES values keeps a sample
    of its rows, in order, drawn from a fixed seed: the same rows at every run with the same arguments."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        keep = max(1, DUMP_VALUES // (a.size // len(a)))
        if len(a) > keep:
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def finish(world, dist):
    """N > 1: leave through a barrier, give destroy_process_group 20 s, then exit the process for good - a
    teardown that hangs after the result line is printed would stall the whole launch."""
    sys.stdout.flush()
    if world <= 1:
        return
    try:
        dist.barrier()
    except Exception:  # noqa: BLE001
        pass
    t = threading.Thread(target=dist.destroy_process_group, daemon=True)
    t.start()
    t.join(20)
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


# ----------------------------------------------------------------------------- B200 arm, 4K tiles
W4K, H4K = 3840, 2160
TILE_COLS_LOG2, TILE_ROWS_LOG2 = 2, 1     # 4 x 2 tiles of 15 x 17 superblocks (BASELINE configs[4])


def run_b200_tiles(args, rank, world, local_rank, embedded=False):
    """BASELINE configs[4]: 4K 8-bit, 8 tiles, speed-6 RDO legs + CDEF, tile t owned by rank t mod N
    (encoder.rs:3249-3257 runs one worker per tile; tiling/tiler.rs:97-132 lays the grid out).  STRONG
    scaling: the job - F 4K frame pairs, every tile of every frame - is the same at every N; a rank
    works on its own tiles of all frames (candidate evaluations only READ the shared reference planes,
    so every rank holds the planes and nothing but the winners is exchanged).  Per step and rank:
      SAD lists (64 / block) + winners, SATD lists (8 / block), residual + 16x16 DCT of the winners -
      one launch each over the F frames - then cdef_find_dir + cdef_filter of the rank's tiles;
      the 8-byte winner records {sad, mv} go to every rank by an NCCL all-gather enqueued on a SIDE
      stream as soon as the SAD leg is done, overlapped with the SATD / transform / CDEF legs.
    The whole step is captured into one CUDA graph (hundreds of tile-sized launches at N = 1)."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    from rav1e_b200 import backend as B
    from rav1e_b200 import shard

    # embedded: called from run_b200 at the end of the 1080p measurement (same process group, own stream
    # and context); returns the result instead of printing it, without the e2e / CPU legs
    torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.Stream(device=local_rank)
    side = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    ctx = B.Context(local_rank, use_torch_stream=True)
    F = args.frames_4k
    tiles = shard.tile_grid(W4K, H4K, TILE_COLS_LOG2, TILE_ROWS_LOG2)
    NT = len(tiles)
    mine = shard.owned_units(NT, rank, world)
    blocks = np.concatenate([shard.blocks_in_rect(tiles[t], BW, BH, B.BLOCK_DTYPE) for t in mine])
    nb = len(blocks)                                       # this rank's blocks per frame
    nb_all = sum(len(shard.blocks_in_rect(t, BW, BH, B.BLOCK_DTYPE)) for t in tiles)
    upr = shard.units_per_rank(NT, world)
    nb_pad = max(len(shard.blocks_in_rect(t, BW, BH, B.BLOCK_DTYPE)) for t in tiles) * upr   # all-gather slot
    # ---- planes: every rank holds every frame (tiles read across their borders)
    uniq = []
    for i in range(min(2, F)):
        rng = np.random.default_rng(4000 + i)
        ref = rng.integers(0, 256, (H4K + 2 * PAD, W4K + 2 * PAD), dtype=np.uint8)
        cur = np.clip(np.roll(ref, (2 - i, -3 + i), axis=(0, 1)).astype(np.int16)
                      + rng.integers(-2, 3, ref.shape, dtype=np.int16), 0, 255).astype(np.uint8)
        uniq.append((cur, ref))
    planes, outs = [], []
    for f in range(F):
        pr = []
        for img in uniq[f % len(uniq)]:
            p = B.Plane()
            ctx.check(ctx.L.b200_plane_alloc(ctx.h, W4K + 2 * PAD, H4K + 2 * PAD, 0, 1, C.byref(p)))
            ctx.check(ctx.L.b200_plane_upload(ctx.h, C.byref(p), img.ctypes.data, img.strides[0]))
            q = B.Plane()
            q.data = p.data + PAD * p.stride + PAD
            q.stride, q.width, q.height, q.pad, q.bpp, q.alloc = p.stride, W4K, H4K, PAD, 1, None
            pr.append(q)
        planes.append(pr)
        outs.append(ctx.plane_alloc(W4K, H4K, 0, 1))       # the frame's CDEF output
    # ---- descriptors of this rank's blocks, frame after frame (b200_*_multi_dev layout)
    n_sad, n_satd = nb * CAND_SAD, nb * CAND_SATD
    sad_np, satd_np = [], []
    for f in range(F):
        c, _ = cand_list(nb, CAND_SAD, 11 * f + 1 + 1000 * rank)
        c["block"] += f * nb
        sad_np.append(c)
        c2, _ = cand_list(nb, CAND_SATD, 11 * f + 2 + 1000 * rank)
        c2["block"] += f * nb
        satd_np.append(c2)
    d_sad_c = torch.from_numpy(np.concatenate(sad_np).view(np.uint8)).cuda()
    d_satd_c = torch.from_numpy(np.concatenate(satd_np).view(np.uint8)).cuda()
    del sad_np, satd_np
    d_blocks_all = torch.from_numpy(np.tile(blocks, F).view(np.uint8)).cuda()
    d_offs = torch.from_numpy((np.arange(F * nb + 1, dtype=np.uint64) * CAND_SAD).astype(np.uint32).view(np.uint8)).cuda()
    d_offs2 = torch.from_numpy((np.arange(F * nb + 1, dtype=np.uint64) * CAND_SATD).astype(np.uint32).view(np.uint8)).cuda()
    d_best = torch.zeros(F * nb * 16, dtype=torch.uint8, device="cuda")
    d_best2 = torch.empty(F * nb * 16, dtype=torch.uint8, device="cuda")
    d_coef = torch.empty(F * nb * BW * BH, dtype=torch.int16, device="cuda")
    pairs = B.PlanePairs([planes[f][0] for f in range(F)], [planes[f][1] for f in range(F)],
                         [(i + 1) * nb for i in range(F)], [(i + 1) * n_sad for i in range(F)])
    pairs2 = B.PlanePairs([planes[f][0] for f in range(F)], [planes[f][1] for f in range(F)],
                          [(i + 1) * nb for i in range(F)], [(i + 1) * n_satd for i in range(F)])
    p_sad = B.me_params(BW, BH, W4K, H4K, LAMBDA, window_hint_px=MV_RANGE_PX)
    p_satd = B.me_params(BW, BH, W4K, H4K, LAMBDA, use_satd=True, window_hint_px=MV_RANGE_PX)
    # CDEF state per frame (frame-indexed arrays; a rank fills the entries of its own tiles)
    n8 = (W4K // 8) * (H4K // 8)
    sbw, sbh = (W4K + 63) // 64, (H4K + 63) // 64
    d_dir = torch.zeros(F * n8, dtype=torch.uint8, device="cuda")
    d_var = torch.zeros(F * n8, dtype=torch.int32, device="cuda")
    d_str = torch.from_numpy(np.random.default_rng(9).integers(0, 64, sbw * sbh).astype(np.uint8)).cuda()
    rects8 = [(tiles[t][0] // 8, tiles[t][1] // 8, tiles[t][2] // 8, tiles[t][3] // 8) for t in mine]
    # winner records: 8 bytes {sad u32, mv_row i16, mv_col i16} = bytes 8..15 of b200_me_result
    rec_local = torch.zeros((F, nb_pad, 8), dtype=torch.uint8, device="cuda")
    gathered = torch.empty((world, F, nb_pad, 8), dtype=torch.uint8, device="cuda") if world > 1 else None
    ev_sad, ev_comm = torch.cuda.Event(), torch.cuda.Event()

    def leg_sad():
        ctx.me_candidates_multi_dev(pairs, d_blocks_all, F * nb, d_sad_c, F * n_sad, p_sad, d_offs, None, None, None, d_best)

    def leg_satd():
        ctx.me_candidates_multi_dev(pairs2, d_blocks_all, F * nb, d_satd_c, F * n_satd, p_satd, d_offs2, None, None, None, d_best2)

    def leg_txfm():
        ctx.fwd_txfm_residual_multi_dev(pairs, d_blocks_all, F * nb, d_best, d_coef, 2, 0, 8)

    # every (frame, owned tile) of the batch as one item list: 32 items per launch
    items = (B.CdefItem * (F * len(rects8)))()
    k = 0
    for f in range(F):
        for r8 in rects8:
            it = items[k]
            it.inp, it.out = C.pointer(planes[f][0]), C.pointer(outs[f])
            it.d_skip8 = None
            it.d_dir, it.d_var = d_dir.data_ptr() + f * n8, d_var.data_ptr() + f * n8 * 4
            it.rx8, it.ry8, it.rw8, it.rh8 = r8
            k += 1

    def leg_cdef_dir():
        ctx.cdef_tiles_dev(items, 0, 0, 0, W4K, H4K, 8, 5, d_str, find_dir=True, filter=False)

    def leg_cdef_filter():
        ctx.cdef_tiles_dev(items, 0, 0, 0, W4K, H4K, 8, 5, d_str, find_dir=False, filter=True)

    def leg_comm():
        """on the side stream: pack the winners to 8-byte records, all-gather them"""
        rec_local[:, :nb].copy_(d_best.view(F, nb, 16)[:, :, 8:16])
        if world > 1:
            dist.all_gather_into_tensor(gathered, rec_local)

    def step_body():
        leg_sad()
        ev_sad.record(stream)
        with torch.cuda.stream(side):
            side.wait_event(ev_sad)
            leg_comm()
            ev_comm.record(side)
        leg_satd()
        leg_txfm()
        leg_cdef_dir()
        leg_cdef_filter()
        stream.wait_event(ev_comm)          # the step is over when the winners have arrived everywhere

    for _ in range(2):                       # eager warm-up (one-time attribute / tensor-map setup)
        step_body()
    torch.cuda.synchronize()
    graph = None
    # NCCL inside a captured graph works, but tearing such a process group down has hung a 2-rank run
    # (and the graph buys ~0: the step is GPU-bound): eager at N > 1 unless --graph asks for it
    if not args.no_graph and (world == 1 or args.graph):
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                step_body()
            g.replay()
            torch.cuda.synchronize()
            graph = g
        except Exception as e:  # noqa: BLE001 - capture is an optimisation, eager is always valid
            sys.stderr.write(f"[bench] CUDA graph capture failed ({type(e).__name__}: {e}); running eagerly\n")
            torch.cuda.synchronize()
    step = (lambda: graph.replay()) if graph is not None else step_body

    def timed(fn, reps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    clk = ClockSampler(local_rank)
    if rank == 0 and not embedded:
        clk.start()
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    l0 = ctx.launches
    step_body() if graph is not None else None     # launch count of one step (graph replays do not count)
    torch.cuda.synchronize()
    launches_per_step = (ctx.launches - l0) if graph is not None else None
    l0 = ctx.launches
    ms = timed(step, args.steps)
    if launches_per_step is None:
        launches_per_step = (ctx.launches - l0) // args.steps
    for _ in range(int(min(2000, max(0, 250.0 / max(ms / args.steps, 1e-3) - args.steps)))):   # ~0.25 s more of the
        step()                                                   # same steps (untimed): clock samples under load
    torch.cuda.synchronize()
    units_per_step = F * nb_all * (CAND_SAD + CAND_SATD + 1)        # the whole job, every tile
    value = units_per_step * args.steps / (ms * 1e-3)
    legs = {}
    for name, fn in (("sad_cand", leg_sad), ("satd_cand", leg_satd), ("residual+fwd_txfm", leg_txfm),
                     ("cdef_find_dir", leg_cdef_dir), ("cdef_filter", leg_cdef_filter)):
        fn()
        legs[name] = timed(fn, max(2, args.steps // 2)) / max(2, args.steps // 2)

    def comm_alone():
        leg_comm()
    comm_alone()
    ms_comm = timed(comm_alone, max(2, args.steps // 2)) / max(2, args.steps // 2)
    clocks = clk.stop() if rank == 0 and not embedded else None
    if embedded:
        res = None
        if rank == 0:
            res = {"workload": "4k-8bit-speed6-8tiles (BASELINE configs[4])", "scaling": "strong",
                   "value": value, "unit": "blocks/s", "ms_per_step": ms / args.steps, "n_gpus": world,
                   "frame_pairs": F, "blocks_per_frame": nb_all, "tiles": NT,
                   "parallelism": f"tile t -> rank t mod {world} ({len(mine)} tile(s) per rank); total work fixed; "
                                  "the N=1 line of the same run series is the baseline",
                   "legs": "64 SAD + 8 SATD candidates + residual/DCT per 16x16 block, cdef_find_dir + cdef_filter per tile "
                           "(CDEF time is in the step, not in the unit count)",
                   "collective": {"what": "NCCL all-gather of 8-byte winner records on a side stream behind the SAD leg",
                                  "bytes_per_rank": int(rec_local.numel()), "ms_alone": ms_comm},
                   "cuda_graph": graph is not None, "per_rank_leg_ms": legs,
                   "gpu_launches": int(launches_per_step * args.steps)}
        graph = step = None
        torch.cuda.synchronize()
        for pl in outs:
            ctx.plane_free(pl)
        return res
    # the same job on ONE GPU is the strong-scaling baseline: rank 0 cannot run it inside an N-rank
    # launch without the other ranks idling, so it is measured by `--gpus 1 --workload 4k-tiles`
    e2e = run_e2e(ctx, grid_blocks(), args, world, dist if world > 1 else None)
    if rank == 0:
        peak, peak_src = peaks()
        alg_bytes = int((F * n_sad * (BW * BH + 4) + F * nb * BW * BH))
        out = {
            "metric": METRIC, "value": value, "unit": "blocks/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "4k-8bit-speed6-8tiles (BASELINE configs[4])", "frame": [W4K, H4K],
                       "tiles": NT, "tile_grid": "4x2 (tile_cols_log2 2, tile_rows_log2 1; 960x1088 / 960x1072 px)",
                       "frame_pairs": F, "blocks_per_frame": nb_all, "block": "16x16",
                       "legs": {"sad_candidates_per_block": CAND_SAD, "satd_candidates_per_block": CAND_SATD,
                                "fwd_txfm_per_block": "1 x TX_16X16 DCT_DCT of the SAD winner's residual",
                                "cdef": "cdef_find_dir + cdef_filter (luma) over every tile; not counted in `value`'s units"},
                       "parallelism": f"tile t -> rank t mod {world} ({len(mine)} tile(s) per rank); total work fixed",
                       "collective": {"what": "NCCL all-gather of 8-byte winner records {sad, mv} per block to every rank, "
                                              "on a side stream after the SAD leg, overlapped with the SATD / transform / CDEF legs",
                                      "bytes_per_rank": int(rec_local.numel()), "ms_alone": ms_comm},
                       "cuda_graph": graph is not None,
                       "l2": "planes %.0f MB on every rank; a rank touches its tiles (1/%d of them)" % (
                           F * 2 * (W4K + 2 * PAD) * (H4K + 2 * PAD) / 1e6, world),
                       "per_rank_leg_ms (rank 0, each leg alone)": legs,
                       "mv_range_px": MV_RANGE_PX, "lambda": LAMBDA},
            "roofline": {"kernel": "me_cand_group_u8<16,16,SAD> over rank 0's tiles of all frames",
                         "bound": "hbm", "achieved": alg_bytes / (legs["sad_cand"] * 1e-3) / 1e9, "peak": peak,
                         "unit": "GB/s", "frac": alg_bytes / (legs["sad_cand"] * 1e-3) / 1e9 / peak, "traffic": None,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                         "launch_ms": legs["sad_cand"]},
            "cpu_baseline": run_cpu_baseline(grid_blocks()), "e2e": e2e, "clocks": clocks,
            "gpu_launches": int(launches_per_step * args.steps),
        }
        print(json.dumps(out))
    graph = step = None          # a captured NCCL node must not outlive its communicator
    torch.cuda.synchronize()
    finish(world, dist)


def run_e2e_lists(ctx0, blocks, args, world=1, dist=None):
    """The same metric through the host-buffer C ABI, one call per frame (b200_frame_pipe_push): the
    frame's visible area travels host->device ONCE from pinned memory (the previously pushed frame is
    the reference), the candidate lists travel as 2-byte full-pel offsets, the SAD winners feed the
    fused residual + 16x16 DCT on the device, and winners + coefficients travel device->host.  Frames
    are pipelined over NCTX contexts (streams) in asynchronous mode, one host thread each (like one
    rayon worker per tile, encoder.rs:3253), so PCIe copies overlap kernels; everything is synchronised
    before the clock stops.  Runs on every rank; the ranks' frames add up, the slowest rank's time
    counts."""
    import torch
    from rav1e_b200 import backend as B
    nb = len(blocks)
    NCTX = int(os.environ.get("B200_E2E_CONTEXTS", "4"))
    # frames per step: the contexts run dry at every step boundary (the clock stops on a full
    # synchronisation), so a step holds enough frames per context for the pipeline to be mostly full
    Fe = int(os.environ.get("B200_E2E_FRAMES_PER_CTX", "8")) * NCTX
    pinned = lambda n, dt=np.uint8: torch.empty(n, dtype=torch.uint8).pin_memory().numpy().view(dt)
    ctxs = [B.Context(ctx0.device) for _ in range(NCTX)]
    pipes = []
    for c in ctxs:
        c.set_async(True)
        pipes.append(B.FramePipe(c, W, H, PAD, (BW, BH), LAMBDA, CAND_SAD, CAND_SATD, MV_RANGE_PX, tx_size=2, tx_type=0))
        assert pipes[-1].nblocks == nb
    frames = []
    n_so, n_to = nb * CAND_SAD * 2, nb * CAND_SATD * 2
    for f in range(Fe):
        cur_img, _ = synth_frame_pair(5000 + (f % 4))
        # one pinned packet per frame: [frame | SAD offsets | SATD offsets] back to back travels as ONE
        # copy; the results come back as one block [SAD winners | SATD winners | coefficients]
        pin = pinned(W * H + n_so + n_to)
        hc = pin[:W * H].reshape(H, W)
        hc[:] = cur_img[PAD:PAD + H, PAD:PAD + W]
        c, _ = cand_list(nb, CAND_SAD, 900 + f)
        c2, _ = cand_list(nb, CAND_SATD, 1900 + f)
        # a search stage's pattern around its predictor: (row, col) full-pel offsets, 2 bytes per candidate
        so = pin[W * H:W * H + n_so].view(np.int8).reshape(len(c), 2)
        so[:, 0], so[:, 1] = c["mv_row"] // 8, c["mv_col"] // 8
        to = pin[W * H + n_so:].view(np.int8).reshape(len(c2), 2)
        to[:, 0], to[:, 1] = c2["mv_row"] // 8, c2["mv_col"] // 8
        pout = pinned(2 * nb * 16 + nb * BW * BH * 2)
        best = pout[:nb * 16].view(B.ME_RESULT_DTYPE)
        best2 = pout[nb * 16:2 * nb * 16].view(B.ME_RESULT_DTYPE)
        coef = pout[2 * nb * 16:].view(np.int16).reshape(nb, BW * BH)
        frames.append((hc, so, to, best, best2, coef))
    for k in range(NCTX):           # each pipe needs a reference before its first timed frame
        pipes[k].push(frames[k][0])
        ctxs[k].synchronize()

    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(NCTX)

    def drive(k):
        """ctypes releases the GIL inside the C ABI, so the CUDA API work of the contexts overlaps."""
        nb_h2d = nb_d2h = 0
        for f in range(k, Fe, NCTX):
            hc, so, to, best, best2, coef = frames[f]
            pipes[k].push(hc, so, to, None, best, best2, coef)
            nb_h2d += hc.nbytes + so.nbytes + to.nbytes
            nb_d2h += best.nbytes + best2.nbytes + coef.nbytes
        ctxs[k].synchronize()
        return nb_h2d, nb_d2h

    h2d = d2h = 0

    def step():
        nonlocal h2d, d2h
        res = list(pool.map(drive, range(NCTX)))
        h2d, d2h = sum(r[0] for r in res), sum(r[1] for r in res)
    for _ in range(2):
        step()
    reps = args.steps
    l0 = sum(cx.launches for cx in ctxs)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    dt = time.perf_counter() - t0
    launches = sum(cx.launches for cx in ctxs) - l0
    if world > 1:       # whole job: every rank's frames, the slowest rank's time
        t = torch.tensor([dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt_job = float(t.item())
    else:
        dt_job = dt
    units = world * Fe * nb * (CAND_SAD + CAND_SATD + 1)
    # what the link itself sustains on this box: pinned host <-> device, 256 MB, CUDA events
    big = torch.empty(256 << 20, dtype=torch.uint8).pin_memory()
    dbig = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def link(dst, src):
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(4):
            dst.copy_(src, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        return 4 * big.numel() / (e0.elapsed_time(e1) * 1e-3) / 1e9
    h2d_gbs, d2h_gbs = link(dbig, big), link(big, dbig)

    def link_bidir():
        """both directions at once, in the e2e's own proportion of bytes (what the pipes ask of the link)"""
        big2 = torch.empty(256 << 20, dtype=torch.uint8).pin_memory()
        dbig2 = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        n_up = 192 << 20
        n_dn = min(int(n_up * (d2h / max(h2d, 1))), 256 << 20)
        su, sd = torch.cuda.Stream(), torch.cuda.Stream()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        with torch.cuda.stream(su):
            ev[0].record()
            for _ in range(4):
                dbig[:n_up].copy_(big[:n_up], non_blocking=True)
            ev[1].record()
        with torch.cuda.stream(sd):
            ev[2].record()
            for _ in range(4):
                big2[:n_dn].copy_(dbig2[:n_dn], non_blocking=True)
            ev[3].record()
        torch.cuda.synchronize()
        return (4 * n_up / (ev[0].elapsed_time(ev[1]) * 1e-3) / 1e9, 4 * n_dn / (ev[2].elapsed_time(ev[3]) * 1e-3) / 1e9)
    h2d_bi, d2h_bi = link_bidir()
    del big, dbig
    res = {"value": units * reps / dt_job, "unit": "blocks/s", "h2d_bytes_per_step": int(h2d) * world,
           "d2h_bytes_per_step": int(d2h) * world, "frames_per_step": Fe * world,
           "kernel_launches_per_step": launches // reps * world,
           "h2d_GBps_achieved": h2d * reps / dt / 1e9, "d2h_GBps_achieved": d2h * reps / dt / 1e9,
           "h2d_GBps_link_measured": h2d_gbs, "d2h_GBps_link_measured": d2h_gbs,
           "h2d_GBps_link_bidirectional": h2d_bi, "d2h_GBps_link_bidirectional": d2h_bi,
           "link_frac": max(h2d * reps / dt / 1e9 / h2d_bi, d2h * reps / dt / 1e9 / d2h_bi), "ranks": world,
           "workload": "1080p-8bit-speed6-me16x16 frames, one stream of frames per rank (per-GPU work fixed)",
           "api": "per frame: ONE b200_frame_pipe_push (frame uploaded once - the previous frame is the reference; "
                  "candidate lists as 2-byte full-pel offsets; SAD winners -> residual + 16x16 DCT on the device; "
                  f"winners + coefficients out); {NCTX} contexts in async mode, one host thread each; "
                  "per-rank link rates shown, bytes and frames summed over ranks"}
    pool.shutdown()
    for c, pp in zip(ctxs, pipes):
        pp.close()
        c.close()
    return res



E2E_DCQ, E2E_ACQ = 88, 100          # quantizer steps of the streamed e2e mode (8-bit; a mid-range qindex)


def run_e2e_stream(ctx0, blocks, args, world=1, dist=None):
    """End to end the way an encoder feeds the device (VERDICT r1 item 3): per frame ONE b200_frame_pipe_push_packed -
    only the NEW FRAME goes host->device (the previous push is the reference; the search patterns are encoder constants,
    uploaded once with b200_frame_pipe_set_lists), the device runs SAD lists -> SATD lists -> residual + 16x16 DCT of the
    SAD winner -> quantize chain, and what comes back is what the entropy coder reads: winners, per-block eob and
    tx-domain distortion, and the eob quantized coefficients of every block in scan order (packed, variable size).
    Same units per frame as the device-resident step (64 + 8 + 1 per block); the quantize chain and the packing are
    extra, uncounted work.  Frames are a low-pass synthetic sequence with small global motion, so that residuals
    quantize like video does (the packed size depends on the content; the bytes are counted from the real totals)."""
    import torch
    from scipy.ndimage import uniform_filter
    from rav1e_b200 import backend as B
    nb = len(blocks)
    NCTX = int(os.environ.get("B200_E2E_CONTEXTS", "6" if world == 1 else "4"))
    Fe = int(os.environ.get("B200_E2E_FRAMES_PER_CTX", "8")) * NCTX
    pinned = lambda n, dt=np.uint8: torch.empty(n, dtype=torch.uint8).pin_memory().numpy().view(dt)
    ctxs = [B.Context(ctx0.device) for _ in range(NCTX)]
    rng = np.random.default_rng(31)
    canvas = rng.integers(0, 256, (H + 128, W + 128)).astype(np.float32)
    for _ in range(2):
        canvas = uniform_filter(canvas, size=9, mode="wrap")
    canvas = (canvas - canvas.min()) / (canvas.max() - canvas.min()) * 255.0
    CAP = nb * 64                                            # packed coefficients a frame may return (25 % of dense)
    pipes, frames = [], []
    for k, c in enumerate(ctxs):
        c.set_async(True)
        pp = B.FramePipe(c, W, H, PAD, (BW, BH), LAMBDA, CAND_SAD, CAND_SATD, MV_RANGE_PX, tx_size=2, tx_type=0,
                         dc_quant=E2E_DCQ, ac_quant=E2E_ACQ)
        assert pp.nblocks == nb
        cs, _ = cand_list(nb, CAND_SAD, 900 + k)
        ct, _ = cand_list(nb, CAND_SATD, 1900 + k)
        so = np.stack([cs["mv_row"] // 8, cs["mv_col"] // 8], axis=1).astype(np.int8)
        to = np.stack([ct["mv_row"] // 8, ct["mv_col"] // 8], axis=1).astype(np.int8)
        pp.set_lists(so, to)
        pipes.append(pp)
    for f in range(Fe):
        hc = pinned(W * H).reshape(H, W)
        dx, dy = (3 * f) % 41, (2 * f) % 29                  # slow global motion
        img = canvas[32 + dy:32 + dy + H, 32 + dx:32 + dx + W] + rng.integers(-1, 2, (H, W))
        hc[:] = np.clip(np.rint(img), 0, 255).astype(np.uint8)
        res = pinned(2 * nb * 16)
        frames.append((hc, res[:nb * 16].view(B.ME_RESULT_DTYPE), res[nb * 16:].view(B.ME_RESULT_DTYPE),
                       pinned(nb * 2).view(np.uint16), pinned(nb * 8).view(np.uint64), pinned(CAP * 2).view(np.int16)))
    for k in range(NCTX):
        pipes[k].push_packed(frames[k][0])
        ctxs[k].synchronize()

    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(NCTX)

    def drive(k):
        up = down = coefs = trunc = 0
        for f in range(k, Fe, NCTX):
            hc, b1, b2, eob, dist, packed = frames[f]
            n = pipes[k].push_packed(hc, b1, b2, eob, dist, packed)
            up += hc.nbytes
            down += b1.nbytes + b2.nbytes + eob.nbytes + dist.nbytes + 4 + 2 * min(n, CAP)
            coefs += n
            trunc += n > CAP
        ctxs[k].synchronize()
        return up, down, coefs, trunc

    tot = [0, 0, 0, 0]

    def step():
        res = list(pool.map(drive, range(NCTX)))
        for q in range(4):
            tot[q] = sum(r[q] for r in res)
    for _ in range(2):
        step()
    reps = args.steps
    l0 = sum(cx.launches for cx in ctxs)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    dt = time.perf_counter() - t0
    launches = sum(cx.launches for cx in ctxs) - l0
    if world > 1:
        t = torch.tensor([dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt_job = float(t.item())
    else:
        dt_job = dt
    units = world * Fe * nb * (CAND_SAD + CAND_SATD + 1)
    h2d, d2h, coefs, trunc = tot
    out = {"value": units * reps / dt_job, "unit": "blocks/s", "h2d_bytes_per_step": int(h2d) * world,
           "d2h_bytes_per_step": int(d2h) * world, "frames_per_step": Fe * world,
           "kernel_launches_per_step": launches // reps * world,
           "h2d_GBps_achieved": h2d * reps / dt / 1e9, "d2h_GBps_achieved": d2h * reps / dt / 1e9,
           "packed_coefficients_per_block": coefs / (Fe * nb), "frames_over_packed_capacity": int(trunc), "ranks": world,
           "quantizer": {"dc_quant": E2E_DCQ, "ac_quant": E2E_ACQ},
           "workload": "1080p-8bit-speed6-me16x16 frame stream per rank (per-GPU work fixed): low-pass synthetic frames "
                       "with small global motion",
           "api": "per frame ONE b200_frame_pipe_push_packed: the new frame up (the previous push is the reference, the "
                  "candidate patterns are resident), SAD lists -> SATD lists -> residual + 16x16 DCT of the SAD winner -> "
                  "quantize chain on the device; winners + eob + tx-domain distortion + the eob quantized coefficients of "
                  f"each block in scan order come back; {NCTX} contexts, one host thread each"}
    pool.shutdown()
    for c, pp in zip(ctxs, pipes):
        pp.close()
        c.close()
    return out


def run_e2e(ctx0, blocks, args, world=1, dist=None):
    """e2e.value = the streamed mode (frame in, packed results out); `dense_lists_mode` = round 1's definition made
    faster (candidate lists up with every frame, the dense coefficient block down), measured in the same run.
    B200_E2E_MODE = stream | lists | both (default both)."""
    mode = os.environ.get("B200_E2E_MODE", "both")
    lists = stream = None
    err = None
    if mode in ("lists", "both"):
        lists = run_e2e_lists(ctx0, blocks, args, world, dist)
    if mode in ("stream", "both"):
        try:
            stream = run_e2e_stream(ctx0, blocks, args, world, dist)
        except Exception as e:  # noqa: BLE001 - the line must come out; the dense mode is then the e2e number
            if world > 1:
                raise           # (ranks must not diverge: a collective sits inside)
            err = f"{type(e).__name__}: {e}"
            if lists is None:
                lists = run_e2e_lists(ctx0, blocks, args, world, dist)
    if stream is None:
        res = dict(lists)
        if err:
            res["stream_mode_error"] = err
        return res
    res = dict(stream)
    if lists is not None:
        res["dense_lists_mode"] = lists
        for k in ("h2d_GBps_link_measured", "d2h_GBps_link_measured", "h2d_GBps_link_bidirectional",
                  "d2h_GBps_link_bidirectional"):
            res[k] = lists[k]
    return res


def run_cpu_baseline(blocks):
    from tests import oracle_lib as O
    threads = O.host_threads()
    cur_img, ref_img = synth_frame_pair(0)
    ocur, oref = O.Plane(W, H, PAD), O.Plane(W, H, PAD)
    ocur.data[:], oref.data[:] = cur_img, ref_img
    sad_c, _ = cand_list(len(blocks), CAND_SAD, 100)
    satd_c, _ = cand_list(len(blocks), CAND_SATD, 200)
    resid = np.random.default_rng(5).integers(-255, 256, (len(blocks), BH, BW)).astype(np.int16)
    O.fullpel_candidates(ocur, oref, blocks, sad_c[:65536], BW, BH, False, LAMBDA)   # warm
    t0 = time.perf_counter()
    reps = 0
    while time.perf_counter() - t0 < 3.0:
        O.fullpel_candidates(ocur, oref, blocks, sad_c, BW, BH, False, LAMBDA, threads=threads)
        O.fullpel_candidates(ocur, oref, blocks, satd_c, BW, BH, True, LAMBDA, threads=threads)
        O.forward_transform_batch(resid, 2, 0, 8, threads=threads)
        reps += 1
    dt = time.perf_counter() - t0
    units = (len(sad_c) + len(satd_c) + len(resid)) * reps
    return {"value": units / dt, "unit": "blocks/s", "cores": threads, "kind": "port",
            "sample": f"1 frame pair x {reps} passes ({CAND_SAD} SAD + {CAND_SATD} SATD cands + 1 fwd txfm per block), "
                      f"{dt:.1f} s wall on {threads} threads; C restatement of rav1e rust:: kernels"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=FRAMES_PER_GPU)
    ap.add_argument("--workload", default="auto", choices=["auto", "1080p", "4k-tiles"],
                    help="auto: BASELINE configs[1] (1080p lookahead batch, per-GPU work fixed: weak scaling) as the "
                         "line's metric at every N, plus configs[4] (4K, 8 tiles sharded over the ranks, total work "
                         "fixed: strong scaling) in `strong_scaling_4k_tiles`; 1080p / 4k-tiles: only that one")
    ap.add_argument("--frames-4k", type=int, default=16, help="4K frame pairs of the tile workload")
    ap.add_argument("--no-graph", action="store_true", help="4k-tiles: launch eagerly instead of replaying a CUDA graph")
    ap.add_argument("--graph", action="store_true", help="4k-tiles at N > 1: capture the step (incl. the NCCL all-gather) in a CUDA graph")
    ap.add_argument("--pairs-per-launch", type=int, default=32,
                    help="frame pairs served by one launch of each leg (b200_*_multi_dev); 1 = a launch per pair")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last 1080p step computed on rank 0 as DIR/<name>.npy "
                         "(float64, at most 64 MB in all): per-candidate SAD and SATD, the SAD and SATD winners "
                         "(cost, distortion, mv_row, mv_col) and the winners' coefficients; the inputs are seeded, so "
                         "runs with the same arguments compare output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload == "4k-tiles"):
        ap.error("--dump-outputs writes the outputs of the b200 arm's 1080p step (--impl b200, --workload auto or 1080p)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly one JSON line: NCCL's own log (the version banner included) goes to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    # (NCCL_DEBUG itself is left as the launcher set it; at VERSION / WARN this NCCL build still prints its
    # one-line version banner on stdout, ahead of the JSON line)
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.workload == "4k-tiles":
        run_b200_tiles(args, rank, world, local_rank)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
