#!/usr/bin/env python
"""bench.py -- keyframes/sec of the loop-closure front-end and pose-graph solve ms on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one batch of KF_PER_STEP = 10 four-view fisheye keyframes through the hot path (BASELINE.json config C3 per
GPU; the default 20 steps time 200 keyframes, SURVEY.md section 8d), each keyframe being
  8 x SuperPoint (640x480, up+down images of 4 directions) + 4 x NetVLAD + 4 stereo cross-check matches
  + add_to_database + inner-product top-k against the keyframe database (10 000 rows x 4096 f32 preloaded)
  + acceptance rule + 4 per-direction cross-check matches against the hit keyframe.
`value`  = keyframes/s with the u8 images already resident in HBM (whole job, all ranks).
`e2e`    = the same through the host-buffer C-ABI call osb_frontend_process: pinned host images in, record + loop
           result back to the host, H2D/D2H inside the timed region.
--dump-outputs DIR: the keyframe records and loop results of the last timed step of `value` (rank 0), one .npy per field.
The images, weights and database are seeded, so the same arguments give the same inputs on every run.
N > 1: one drone per GPU (weak scaling); every step ends with ONE NCCL all-gather of the fixed-size keyframe
record (replaces LoopNet's LCM multicast) and each GPU ingests the N-1 foreign records into its remote database.
The pose-graph solve (BASELINE config C5 graph: 2000 nodes / 12 000 factors) is single-GPU ("replicas only"): it is
timed once per run on every rank and reported as `solve_ms`.
`--impl reference`: the reference's CPU path restated by oracle/ (torch CPU SuperPoint/NetVLAD with all host threads,
numpy scan, cross-check matcher, scipy sparse LM) -- the reference itself cannot be built here (DESIGN.md).  With
--gpus N it runs N CPU drones side by side (N processes sharing the host threads), the same weak-scaling workload.
`trt_like_baseline` (N = 1, in the main line): baseline/trt_like.py, the reference's TensorRT structure with the engines
replaced by PyTorch/cuDNN fp16 -- batch 1, H2D + enqueue + D2H of every binding + synchronize per image, CPU
post-processing -- timed on the same GPU and host.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, N_DIRS, MAX_NUM = 640, 480, 4, 200
DB_ROWS = 10000
POOL = 8                      # distinct keyframes cycled through; the first POOL_IN_DB are in the database beforehand (their
POOL_IN_DB = 4                # queries hit from the start), the others are new the first time and revisits afterwards
KF_PER_STEP = 10              # keyframes per step: --steps 20 times 200 keyframes
HOST_ISSUE_KF, STAGE_KF, REPLAY_KF = 8, 5, 120      # keyframes of the untimed / replay passes through the same front-end


def keyframe_rounds(steps: int, warmup: int) -> int:
    """keyframe rounds that go through the main front-end in one run: both timed regions (resident and end to end, warm-up
    included), the host-issue and stage-profile passes, the C4 replay"""
    return 2 * (warmup + steps) * KF_PER_STEP + HOST_ISSUE_KF + STAGE_KF + REPLAY_KF


def db_capacity(db_rows: int, world: int, steps: int, warmup: int) -> int:
    """rows per store: the preloaded rows plus what the run can add -- per round 4 own rows (local store) and 4 rows of every
    other drone (remote store) -- with the host's conservative bound in mind, which charges every gathered record, the
    skipped own slot included, to BOTH stores ((world + 1) * 4 per round), so that it never has to synchronise to find out
    that there is room.  (An undersized store made an 8-rank run fail in its replay leg.)"""
    return db_rows + N_DIRS * (world + 1) * (keyframe_rounds(steps, warmup) + 64) + 1024
SP_GFLOP_PER_IMAGE = 52.10    # SURVEY.md section 8d / BASELINE.md section 2


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--db-rows", type=int, default=DB_ROWS)
    p.add_argument("--no-solve", action="store_true")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-trt-like", action="store_true")
    p.add_argument("--blocking-exchange", action="store_true",
                   help="N > 1: all-gather of round i between extract and ingest of round i (the r01 pipeline), for A/B")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="write the keyframe records and loop results of the last timed step to DIR/<field>.npy")
    p.add_argument("--cpu-drone", type=int, default=-1, help=argparse.SUPPRESS)      # internal: one CPU drone of --impl reference
    p.add_argument("--cpu-threads", type=int, default=0, help=argparse.SUPPRESS)
    a = p.parse_args()
    if a.steps < 1 or a.warmup < 0:
        p.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs writes what the CUDA path computes: --impl ours only")
    return a


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index, self.first = [], None, index, 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 5.0:      # nvidia-smi needs ~1 s before the first sample
                time.sleep(0.05)
        except Exception:
            self.proc = None

    def mark(self):
        """samples taken from now on belong to the timed region"""
        self.first = len(self.rows)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = self.rows[self.first:] if len(self.rows) - self.first >= 2 else self.rows
        sm = [float(r[0]) for r in rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def keyframe_images(seed):
    from omniswarm_b200 import synth
    up = np.stack([synth.image(1000 * seed + d, H, W) for d in range(N_DIRS)])
    down = np.stack([synth.image(1000 * seed + 100 + d, H, W) for d in range(N_DIRS)])
    return up, down


# ----------------------------------------------------------------------------------------------------------------
# CPU path (oracle): used for cpu_baseline (bounded sample) and for --impl reference
# ----------------------------------------------------------------------------------------------------------------
def cpu_keyframe(oracle_state, up, down):
    """One keyframe through the oracle, mirroring the reference call order (loop_cam.cpp:341-523 + loop_detector)."""
    from oracle import frontend_ref as fr
    w, nvw, comp, mean, db, det = oracle_state
    descs = []
    for d in range(N_DIRS):
        u = up[d].copy(); u[H * 3 // 4:] = 0
        dn = down[d].copy(); dn[H * 3 // 4:] = 0
        ku, du, _, _ = fr.superpoint_inference(u, w, 0.015, MAX_NUM, comp, mean)
        kd, dd, _, _ = fr.superpoint_inference(dn, w, 0.015, MAX_NUM, comp, mean)
        g = fr.netvlad_net(u, nvw)
        fr.bf_crosscheck(du, dd)
        descs.append((du, g))
    q = descs[1][1]
    scores = db @ q                                  # faiss::IndexFlatIP scan (BLAS sgemv)
    top = np.argsort(-scores, kind="stable")[:10]
    for d in range(N_DIRS):                          # per-direction match against the hit
        fr.bf_crosscheck(descs[d][0], descs[(d + 1) % N_DIRS][0])
    return int(top[0])


def best_cpu_threads():
    """torch's CPU convolutions do not scale to every core of a 100+ core host: time one SuperPoint image at a few
    thread counts and keep the fastest ("all the host threads it can use")."""
    import torch
    from omniswarm_b200 import synth
    from oracle import frontend_ref as fr
    cores = os.cpu_count() or 1
    w = synth.superpoint_weights(0)
    img = synth.image(0)
    best, best_t = 1, float("inf")
    for t in sorted({min(cores, c) for c in (8, 16, 32, 64, cores)}):
        torch.set_num_threads(t)
        fr.superpoint_net(img, w)
        t0 = time.perf_counter()
        fr.superpoint_net(img, w)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = t, dt
    torch.set_num_threads(best)
    return best, cores


def cpu_baseline(args, n_keyframes=2):
    import torch
    from omniswarm_b200 import synth
    from oracle import solver_ref as sr
    threads, cores = best_cpu_threads()
    comp, mean = synth.pca_matrices(0)
    state = (synth.superpoint_weights(0), synth.netvlad_weights(0), comp, mean,
             synth.descriptor_db(args.db_rows, 4096, 1), None)
    up, down = keyframe_images(0)
    cpu_keyframe(state, up, down)                    # warm-up (thread pools, allocator)
    t0 = time.perf_counter()
    for i in range(n_keyframes):
        cpu_keyframe(state, up, down)
    dt = (time.perf_counter() - t0) / n_keyframes
    out = dict(value=1.0 / dt, unit="keyframes/s", cores=threads, host_cores=cores, kind="port",
               sample=f"{n_keyframes} keyframes (8 SuperPoint + 4 NetVLAD 640x480 via torch CPU fp32, {threads} threads "
                      f"= fastest of 8/16/32/64/{cores}; "
                      f"numpy scan of {args.db_rows} rows; cross-check matcher); reference sets 1 thread "
                      f"(superpoint_tensorrt.cpp:98)")
    if not args.no_solve:
        g = synth.pose_graph_c5(0)
        t0 = time.perf_counter()
        res = sr.solve_fast(g)
        out["solve_ms"] = (time.perf_counter() - t0) * 1e3
        out["solve_iterations"] = int(res["iterations"])
        out["solve_final_cost"] = float(res["final_cost"])
        out["solve_kind"] = "Ceres stand-in: scipy SuperLU (symmetric mode, MMD) LM, Ceres-default tolerances, 1 thread"
    return out


def _cpu_drone(args):
    """one CPU drone of the reference arm: `steps` keyframes on `cpu_threads` torch threads; prints its wall time"""
    import torch
    from omniswarm_b200 import synth
    torch.set_num_threads(max(1, args.cpu_threads))
    comp, mean = synth.pca_matrices(0)
    state = (synth.superpoint_weights(0), synth.netvlad_weights(0), comp, mean,
             synth.descriptor_db(args.db_rows, 4096, 1 + args.cpu_drone), None)
    frames = [keyframe_images(100 * args.cpu_drone + s) for s in range(2)]
    for i in range(max(1, args.warmup)):
        cpu_keyframe(state, *frames[i % len(frames)])
    t0 = time.perf_counter()
    for i in range(args.steps):
        cpu_keyframe(state, *frames[i % len(frames)])
    _JSON_OUT.write(json.dumps({"drone": args.cpu_drone, "wall_s": time.perf_counter() - t0, "keyframes": args.steps}) + "\n")
    _JSON_OUT.flush()


def trt_like_baseline(args, frames, n_keyframes=6):
    """baseline/trt_like.py on the same GPU and host: the reference's TensorRT call structure with cuDNN fp16 engines"""
    import torch
    from omniswarm_b200 import synth
    from baseline.trt_like import TrtLikeFrontend
    torch.set_num_threads(1)                         # the reference pins libtorch to one thread (superpoint_tensorrt.cpp:98)
    comp, mean = synth.pca_matrices(0)
    fe = TrtLikeFrontend(synth.superpoint_weights(0), synth.netvlad_weights(0), comp, mean,
                         synth.descriptor_db(args.db_rows, 4096, 1), H, W, 0.015, MAX_NUM)
    for i in range(3):                               # warm-up: cuDNN autotune, allocator
        fe.keyframe(*frames[i % len(frames)])
    fe.bytes_h2d = fe.bytes_d2h = 0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(n_keyframes):
        hit, nk, nm = fe.keyframe(*frames[i % len(frames)])
    dt = (time.perf_counter() - t0) / n_keyframes
    return {"value": 1.0 / dt, "unit": "keyframes/s", "ms_per_keyframe": dt * 1e3, "kind": "TRT-like stand-in (PyTorch/cuDNN fp16, "
            "channels-last, batch 1; H2D + enqueue + D2H of semi/desc + synchronize per image; CPU NMS2 in C, libtorch "
            "grid_sample/PCA on 1 thread, cv2 BFMatcher, numpy sgemv scan)", "keyframes": n_keyframes,
            "h2d_bytes_per_keyframe": fe.bytes_h2d // n_keyframes, "d2h_bytes_per_keyframe": fe.bytes_d2h // n_keyframes,
            "n_kpts": nk, "note": "end to end from host images to host results, like `e2e`; mirrors "
            "tensorrt_generic.cpp:58-75 + superpoint_tensorrt.cpp:117-230 + loop_cam.cpp:341-523; TensorRT itself is not installable here"}


def run_reference(args):
    if args.cpu_drone >= 0:
        return _cpu_drone(args)
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_all = time.perf_counter()
    n = max(1, args.gpus)
    best, host_cores = best_cpu_threads()
    threads = max(1, min(best, host_cores // n))
    steps = max(1, min(args.steps, 6))               # bounded sample: a CPU keyframe takes seconds
    warm = max(1, min(args.warmup, 1))
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT")}
    env["CUDA_VISIBLE_DEVICES"] = ""                 # the arm must not touch a GPU
    procs = [subprocess.Popen([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--cpu-drone", str(d),
                               "--cpu-threads", str(threads), "--steps", str(steps), "--warmup", str(warm),
                               "--db-rows", str(args.db_rows)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, env=env)
             for d in range(n)]
    walls = []
    for p in procs:
        out, _ = p.communicate()
        walls.append(json.loads(out.strip().splitlines()[-1])["wall_s"])
    dt = max(walls) / steps                          # N drones run side by side: the slowest one bounds the swarm
    val = n / dt
    sample = (f"bounded sample: {steps} keyframes per drone (a step of the GPU arm is {KF_PER_STEP} keyframes; ms_per_step is "
              f"scaled to that), {n} CPU drone process(es) x {threads} torch threads on a {host_cores}-thread host "
              f"(single-drone optimum: {best} threads, fastest of 8/16/32/64/all); torch CPU fp32 SuperPoint/NetVLAD, numpy "
              f"scan, cross-check matcher: oracle port of the reference path; TensorRT/Ceres are not installable here")
    line = {"impl": "reference", "metric": "keyframes/sec (SuperPoint+NetVLAD+match)", "value": val, "unit": "keyframes/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3 * KF_PER_STEP,
            "keyframes_timed": steps, "ms_per_keyframe": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, n),
            "cpu_baseline": {"value": val, "unit": "keyframes/s", "cores": threads * n, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "keyframes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "cpu_drones": n, "wall_s": time.perf_counter() - t_all}
    _emit(line)


def workload_config(args, world, keyframes_per_step=KF_PER_STEP):
    return {"workload": "C3: 4-view fisheye keyframe (8x SuperPoint 640x480 + 4x NetVLAD + stereo match + DB add + "
                        f"IP top-k vs {args.db_rows}-row x 4096 f32 DB + rule + 4 local matches)",
            "keyframes_per_step": keyframes_per_step, "distinct_keyframes": POOL,
            "images_per_keyframe": 2 * N_DIRS, "db_rows": args.db_rows, "max_kpts": MAX_NUM, "sp_thres": 0.015,
            "parallelism": f"drone-per-GPU x{world}" + (" + 1 NCCL all-gather of the keyframe record per step" if world > 1 else ""),
            "l2_note": "per-step working set (activations ~1.3 GB + DB 164 MB) exceeds the 126 MB L2; no explicit flush"}


# ----------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from omniswarm_b200 import lib, synth, host, swarm

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback in the product path)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    L = lib.load()
    pk = peaks()
    comp, mean = synth.pca_matrices(0)
    spw = synth.flatten_sp_weights(synth.superpoint_weights(0))
    nvw = synth.flatten_nv_weights(synth.netvlad_weights(0))
    # database capacity: the preloaded rows plus everything this run will add.  Every keyframe round adds 4 rows per drone
    # (own -> local store, foreign -> remote store), and the rounds are: both timed regions (warm-up included), the host-issue
    # and stage-profile passes and the C4 replay.  (An undersized store made the 8-rank run fail in the replay leg.)
    fe = host.KeyframeFrontend(spw, comp, mean, nvw, width=W, height=H, n_dirs=N_DIRS, max_num=MAX_NUM, sp_thres=0.015,
                               self_id=rank, db_capacity=db_capacity(args.db_rows, world, args.steps, args.warmup),
                               inner_product_thres=0.3,
                               match_index_dist=5, zero_bottom_quarter=True, accept_min_3d_pts=10)
    st = torch.cuda.current_stream().cuda_stream

    # ---- set-up (untimed): image pool in pinned host memory and in HBM; database preload ----
    frames = [keyframe_images(100 * rank + s) for s in range(POOL)]
    pin_up = [torch.from_numpy(f[0]).pin_memory() for f in frames]
    pin_dn = [torch.from_numpy(f[1]).pin_memory() for f in frames]
    dev_up = [t.cuda() for t in pin_up]
    dev_dn = [t.cuda() for t in pin_dn]
    rec_dev = torch.zeros(lib.RECORD_BYTES, dtype=torch.uint8, device="cuda")
    res_dev = torch.zeros(lib.RESULT_BYTES, dtype=torch.uint8, device="cuda")
    # the resident path writes keyframe k of a step to slot k, so after a step the slots hold everything it computed (N > 1:
    # the asynchronous exchange reads a record one round later; a slot is rewritten only KF_PER_STEP rounds later)
    rec_slots = [torch.zeros(lib.RECORD_BYTES, dtype=torch.uint8, device="cuda") for _ in range(KF_PER_STEP)]
    res_slots = [torch.zeros(lib.RESULT_BYTES, dtype=torch.uint8, device="cuda") for _ in range(KF_PER_STEP)]
    gathered = torch.zeros(world * lib.RECORD_BYTES, dtype=torch.uint8, device="cuda") if world > 1 else None
    # N > 1: the exchange goes through the C ABI (osb_swarm_*: ncclAllGather on the library's own communicator); the
    # 128-byte communicator id travels over the torch.distributed group that also carries the timing reductions
    sw, rec2, gath2, pending = None, None, None, [False]
    if world > 1:
        uid = torch.zeros(lib.SWARM_ID_BYTES, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(host.Swarm.unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        sw = host.Swarm(bytes(uid.cpu().numpy().tobytes()), rank, world)
        rec2 = [torch.zeros(lib.RECORD_BYTES, dtype=torch.uint8, device="cuda") for _ in range(2)]
        gath2 = [torch.zeros(world * lib.RECORD_BYTES, dtype=torch.uint8, device="cuda") for _ in range(2)]
    rec_host = torch.zeros(lib.RECORD_BYTES, dtype=torch.uint8).pin_memory()
    res_host = torch.zeros(lib.RESULT_BYTES, dtype=torch.uint8).pin_memory()
    # the pool keyframes go into the database first (so that every timed query is a revisit that hits), then
    # random unit-norm rows with local descriptors up to db_rows
    for i in range(POOL_IN_DB):
        fe.extract(dev_up[i].data_ptr(), dev_dn[i].data_ptr(), 10_000 + i, rec_dev.data_ptr(), st, device_images=True)
        fe.ingest_own(rec_dev.data_ptr(), st)
    fe.finish(st)
    n_fill = args.db_rows - fe.db_size(False)
    chunk = 2000
    for s in range(0, n_fill, chunk):
        n = min(chunk, n_fill - s)
        g = synth.descriptor_db(n, 4096, 50 + s + 7919 * rank)
        ld = np.random.default_rng(s + rank).standard_normal((n, MAX_NUM, 64)).astype(np.float32)
        fe.db_load(g, ld, np.full(n, MAX_NUM, np.int32), remote=False)
    db_rows_start = fe.db_size(False)

    def swarm_round(i, rec):
        """after extract of keyframe i into `rec`: database work + the ONE collective of the path.
        Default (asynchronous, like the reference's LCM thread, loop_net.cpp:142-172): the own keyframe goes to the local
        database at once, the foreign records of the PREVIOUS round -- whose all-gather ran behind this keyframe's
        extraction -- go to the remote database, and this round's all-gather starts on the library's side stream."""
        if args.blocking_exchange:
            sw.exchange(rec.data_ptr(), gathered.data_ptr(), st)
            fe.ingest(gathered.data_ptr(), world, -1, st)
            return
        b = i & 1
        fe.ingest_own(rec.data_ptr(), st)                                     # add_to_database of the own keyframe
        if pending[0]:
            sw.wait(st)
            fe.ingest(gath2[b ^ 1].data_ptr(), world, rank, st)               # last round's foreign keyframes (own slot skipped)
        sw.exchange_async(rec.data_ptr(), gath2[b].data_ptr(), st)
        pending[0] = True

    def keyframe_resident(i):
        j = i % POOL
        rec, res = rec_slots[i % KF_PER_STEP], res_slots[i % KF_PER_STEP]
        fe.extract(dev_up[j].data_ptr(), dev_dn[j].data_ptr(), i, rec.data_ptr(), st, device_images=True)
        if world > 1:
            swarm_round(i, rec)
        else:
            fe.ingest_own(rec.data_ptr(), st)
        fe.query(rec.data_ptr(), res.data_ptr(), st)

    def keyframe_e2e(i):
        j = i % POOL
        if world == 1:
            fe.process_raw(pin_up[j].data_ptr(), pin_dn[j].data_ptr(), i, rec_host.data_ptr(), res_host.data_ptr())
        else:
            rec = rec2[i & 1]
            fe.extract(pin_up[j].data_ptr(), pin_dn[j].data_ptr(), i, rec.data_ptr(), st)
            swarm_round(i, rec)
            fe.query(rec.data_ptr(), res_dev.data_ptr(), st)
            rec_host.copy_(rec, non_blocking=True); res_host.copy_(res_dev, non_blocking=True)
            fe.finish(st)

    def step_resident(i):                 # one step = one batch of KF_PER_STEP keyframes
        for k in range(KF_PER_STEP):
            keyframe_resident(i * KF_PER_STEP + k)

    def step_e2e(i):
        for k in range(KF_PER_STEP):
            keyframe_e2e(i * KF_PER_STEP + k)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host_issue = [0.0]

    def timed(fn, steps, warmup, base, sampler=None):
        for i in range(warmup):
            fn(base + i)
        fe.finish(st)
        barrier()
        if sampler:
            sampler.mark()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = host.launch_count()
        e0.record()
        for i in range(steps):
            fn(base + warmup + i)
        e1.record()
        fe.finish(st)
        barrier()
        ms = e0.elapsed_time(e1)
        launches = host.launch_count() - l0
        if world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches

    # ---- timed region 1: images resident in HBM ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_total, launches = timed(step_resident, args.steps, args.warmup, 0, sampler)
    last_step = (torch.stack(rec_slots).cpu().numpy(), torch.stack(res_slots).cpu().numpy()) if args.dump_outputs else None
    # host cost of ENQUEUEING a keyframe with an empty launch queue (8 keyframes right after a synchronisation: no back-pressure)
    fe.finish(st); barrier()
    th = time.perf_counter()
    for k in range(HOST_ISSUE_KF):
        keyframe_resident(900_000 + k)
    host_issue_resident = (time.perf_counter() - th) * 1e3 / HOST_ISSUE_KF
    fe.finish(st); barrier()
    clocks = sampler.stop()
    ms_step = ms_total / args.steps
    ms_keyframe = ms_step / KF_PER_STEP
    value = world * 1e3 / ms_keyframe

    # ---- timed region 2: end to end through the host-buffer call (wall clock == device time: sync on both sides) ----
    barrier()
    for i in range(args.warmup):
        step_e2e(5_000 + i)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step_e2e(6_000 + i)
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = world * args.steps * KF_PER_STEP / e2e_s
    res = lib.LoopResult.from_buffer_copy(res_host.numpy().tobytes())
    rec = lib.KeyframeRecord.from_buffer_copy(rec_host.numpy().tobytes())

    # ---- stage breakdown (CUDA events inside the library, one extra profiled pass; not part of `value`) ----
    fe.set_profiling(True)
    stage_acc = {}
    for i in range(STAGE_KF):
        keyframe_resident(700_000 + i)
        fe.finish(st)
        for k, v in fe.stage_ms().items():
            stage_acc.setdefault(k, []).append(v)
    fe.set_profiling(False)
    stages = {k: float(np.median(v)) for k, v in stage_acc.items()}
    db_rows_now = fe.db_size(False)
    db_rows_remote = fe.db_size(True)

    # ---- the collective alone: one blocking all-gather of the 286 KB record, CUDA events, max over ranks ----
    exchange = None
    if world > 1:
        sw.wait(st)
        for _ in range(5):
            sw.exchange(rec2[0].data_ptr(), gathered.data_ptr(), st)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 50
        e0.record()
        for _ in range(reps):
            sw.exchange(rec2[0].data_ptr(), gathered.data_ptr(), st)
        e1.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / reps * 1e3], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        us = float(t.item())
        exchange = {"exchange_us": us, "bytes_per_rank": lib.RECORD_BYTES,
                    "recv_gbs_per_gpu": (world - 1) * lib.RECORD_BYTES / us / 1e3,
                    "frac_of_nvlink_770gbs": (world - 1) * lib.RECORD_BYTES / us / 1e3 / 770.0,
                    "pipeline": "blocking between extract and ingest" if args.blocking_exchange else
                                "asynchronous: round i's ncclAllGather (osb_swarm_exchange_async, side stream) runs behind the "
                                "extraction of keyframe i+1; its foreign records are ingested one round later",
                    "async_transport": sw.transport,
                    "api": "osb_swarm_* (C ABI; exchange_us times the blocking ncclAllGather form)"}

    # ---- rooflines ----
    # dominant kernel: the conv1b launch of conv_umma_kernel<64> (43 % of the network's FLOPs).  Its own duration comes
    # from CUDA events recorded around every layer launch on the library's stream (osb_superpoint_layer_ms).
    GMAC = {"conv1a": 0.17695, "conv1b+pool": 11.3246, "conv2a": 2.83116, "conv2b+pool": 2.83116, "conv3a": 1.41558,
            "conv3b+pool": 2.83116, "conv4a": 0.70779, "conv4b": 0.70779, "convPa": 1.41558, "convPb": 0.07987,
            "convDa": 1.41558, "convDb": 0.31457}          # per 640x480 image, sums to 26.05 (SURVEY.md section 8a)
    sp_prof = host.SuperPoint(spw, comp, mean, W, H, 0.015, MAX_NUM, max_batch=2 * N_DIRS)
    imgs8 = np.concatenate([frames[0][0], frames[0][1]])
    sp_prof.layer_ms(imgs8)
    runs = [sp_prof.layer_ms(imgs8) for _ in range(5)]
    layer_ms = {k: float(np.median([r[k] for r in runs])) for k in runs[0]}
    _c = sp_prof.read("counts").tolist()
    kp_counts = {"candidates": _c[0], "survivors": _c[1], "nms_rounds": _c[2], "phase_cycles": _c[4:8]}
    sp_prof.close()
    layer_tflops = {k: (2 * GMAC[k] * 2 * N_DIRS / v if v > 0 else None) for k, v in layer_ms.items()}
    conv_ms = float(sum(layer_ms.values()))      # the 12 conv launches of a standalone handle (no overlapped work)
    conv_tflops = 2 * N_DIRS * SP_GFLOP_PER_IMAGE / conv_ms  # GFLOP / ms = TFLOP/s
    dom = "conv1b+pool"        # with the default fused first layers this launch is conv1a + conv1b + pool
    dom_gmac = GMAC["conv1a"] + GMAC["conv1b+pool"] if layer_ms["conv1a"] < 0.02 else GMAC["conv1b+pool"]
    dom_tflops = 2 * dom_gmac * 2 * N_DIRS / layer_ms[dom]
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath))
    scan_ms = stages["db_scan"]
    scan_bytes = (db_rows_now + db_rows_remote) * 4096 * 4.0        # local + remote database, each row read once
    scan_gbs = scan_bytes / scan_ms / 1e6
    roofline = {"kernel": "conv1_fused_kernel (conv1a 1->64 computed in the SM by 6 producer warps (lane = pixel, constant-bank weights, FFMA2) + conv1b 64->64 3x3 @640x480 on "
                          "tcgen05 from ONE shared-memory halo copy (9 descriptor views) + fused 2x2 max-pool; split-fp16: hi*hi + "
                          "hi*lo as one MMA of width 128, lo*hi as one of width 64 per K step)",
                "bound": "tensor", "achieved": dom_tflops, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                "frac": dom_tflops / pk["bf16_tflops_sustained"],
                "traffic": (traffic or {}).get("conv1_fused_dram_bytes_per_launch"),
                "algorithmic": f"{2 * N_DIRS} images x {2 * dom_gmac:.3f} GFLOP (conv1a + conv1b, fp32-equivalent MACs x 2); the "
                               "tensor pipes execute 3x conv1b's share as fp16 MACs for fp32-level accuracy",
                "algorithmic_dram_bytes": 2 * N_DIRS * (W * H + (W // 2) * (H // 2) * 64 * 4),
                "ms_per_launch": layer_ms[dom], "mma_tflops_executed": 3 * 2 * GMAC["conv1b+pool"] * 2 * N_DIRS / layer_ms[dom],
                "mma_frac_of_peak": 3 * 2 * GMAC["conv1b+pool"] * 2 * N_DIRS / layer_ms[dom] / pk["bf16_tflops_sustained"],
                "peak_source": pk["source"] + " (sustained: kernel timed inside a long step)"}
    roofline_stack = {"what": "whole SuperPoint conv stack (12 conv launches, per-layer CUDA-event times of a standalone handle)", "achieved": conv_tflops,
                      "unit": "TFLOP/s", "frac": conv_tflops / pk["bf16_tflops_sustained"], "ms": conv_ms,
                      "layer_ms": layer_ms, "layer_tflops": layer_tflops, "keypoint_counts_image0": kp_counts}
    scan_kernel = "db_scan_coop_kernel<1>" if db_rows_now <= 2 * 148 * 64 else "db_scan_kernel<1,4>"
    roofline_match = {"kernel": scan_kernel, "bound": "hbm", "achieved": scan_gbs, "peak": pk["hbm_gbs"],
                      "unit": "GB/s", "frac": scan_gbs / pk["hbm_gbs"],
                      "traffic": (traffic or {}).get("db_scan_dram_bytes_per_launch"),
                      "algorithmic": f"({db_rows_now} local + {db_rows_remote} remote) rows x 16384 B", "ms": scan_ms,
                      "peak_source": pk["source"],
                      "note": "ms = the db_scan stage of a keyframe: the remote-database and the local-database scan launches "
                              "(the merge is fused into each scan's last CTA)"}

    # ---- database scan alone (the HBM-roofline kernel): 10 k rows (config C3) and 50 k rows (config C5) ----
    match_sweep = []
    if rank == 0:
        for rows in (10_000, 50_000):
            idx = host.IndexFlatIP(4096, capacity=rows)
            blk = torch.randn(2000, 4096, device="cuda")
            blk /= blk.norm(dim=1, keepdim=True)
            for s0 in range(0, rows, 2000):
                idx.add_dev(blk.data_ptr(), min(2000, rows - s0), st)
            qd = blk[:1].contiguous()
            sc = torch.empty(1, 10, device="cuda"); ids = torch.empty(1, 10, dtype=torch.int64, device="cuda")
            for _ in range(3):
                idx.search_dev(qd.data_ptr(), 1, 10, sc.data_ptr(), ids.data_ptr(), st)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 20
            e0.record()
            for _ in range(reps):
                idx.search_dev(qd.data_ptr(), 1, 10, sc.data_ptr(), ids.data_ptr(), st)
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / reps
            gbs = rows * 16384 / ms / 1e6
            match_sweep.append({"db_rows": rows, "ms_per_search": ms, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / pk["hbm_gbs"],
                                "note": "scan + merge launches, 1 query, k = 10; "
                                        + ("164 MB > 126 MB L2" if rows == 10_000 else "819 MB >> L2")})
            idx.close(); del blk

    # ---- config C2: one pinhole stream, the reference's own call pattern (one synchronous inference() per image,
    #      host buffers in and out) -- SuperPoint + NetVLAD on a single 640x480 frame ----
    c2 = None
    if rank == 0:
        sp1 = host.SuperPoint(spw, comp, mean, W, H, 0.015, MAX_NUM, max_batch=1)
        nv1 = host.NetVLAD(nvw, W, H, max_batch=1)
        img1 = np.ascontiguousarray(frames[0][0][0])
        for _ in range(3):
            sp1.inference(img1); nv1.inference(img1)
        reps = 40
        t0 = time.perf_counter()
        for _ in range(reps):
            kp1, _d1 = sp1.inference(img1); nv1.inference(img1)
        dt = (time.perf_counter() - t0) / reps
        c2 = {"workload": "C2: single 640x480 pinhole frame, SuperPoint.inference + NetVLAD.inference, host buffers, synchronous",
              "frames_per_s": 1.0 / dt, "ms_per_frame": dt * 1e3, "n_kpts": int(len(kp1))}
        sp1.close(); nv1.close()

    # ---- geometric filter (SURVEY 8f-1): homography-RANSAC masks of the 4 direction pairs of a keyframe, 200 matches each ----
    geometry = None
    if rank == 0:
        rng = np.random.default_rng(3)
        src = rng.uniform(0, 640, (4, 200, 2)).astype(np.float32); src[..., 1] *= 0.75
        dst = src + rng.normal(0, 0.3, src.shape).astype(np.float32) + np.float32(5.0)
        dst[:, ::4] += np.float32(40.0)                                     # 25 % outliers
        t_src, t_dst = torch.from_numpy(src).cuda(), torch.from_numpy(dst).cuda()
        t_n = torch.full((4,), 200, dtype=torch.int32, device="cuda")
        t_mask = torch.zeros(4, 200, dtype=torch.uint8, device="cuda")
        t_inl = torch.zeros(4, dtype=torch.int32, device="cuda"); t_win = torch.zeros(4, dtype=torch.int32, device="cuda")

        def _geo():
            lib.check(L.osb_homography_ransac_dev(C.c_void_p(t_src.data_ptr()), C.c_void_p(t_dst.data_ptr()),
                                                  C.c_void_p(t_n.data_ptr()), 4, 200, C.c_float(3.0), 0,
                                                  C.c_void_p(t_mask.data_ptr()), C.c_void_p(t_inl.data_ptr()),
                                                  C.c_void_p(t_win.data_ptr()), C.c_void_p(st)))
        for _ in range(3):
            _geo()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(50):
            _geo()
        e1.record(); torch.cuda.synchronize()
        geometry = {"what": "osb_homography_ransac_dev: 4 direction pairs x 200 matches, 512 hypotheses each (fp64, "
                            "bit-exact against oracle/geometry_ref.py)", "us_per_keyframe": e0.elapsed_time(e1) / 50 * 1e3,
                    "inliers": t_inl.cpu().tolist()}

    # ---- the stages around the solve and the match that SURVEY 8f lists (rank 0): PCM outlier rejection, PnP-RANSAC + checks,
    #      stereo triangulation -- device time through the _dev entry points ----
    widen = None
    if rank == 0:
        widen = {}
        try:
            edges = synth.pcm_edges(400, 0.35, 1)
            arr = (lib.LoopEdge * len(edges))()
            for i, e in enumerate(edges):
                a = arr[i]
                a.id_a, a.id_b, a.len_a, a.len_b = int(e["id_a"]), int(e["id_b"]), float(e["len_a"]), float(e["len_b"])
                a.rel_pose[:] = [float(x) for x in e["rel"]]; a.cov[:] = [float(x) for x in np.asarray(e["cov"]).reshape(-1)]
                a.odom_a[:] = [float(x) for x in e["odom_a"]]; a.odom_b[:] = [float(x) for x in e["odom_b"]]
            t_e = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).cuda()
            t_c = torch.zeros(len(edges) + 1, dtype=torch.int32, device="cuda")

            def _pcm():
                lib.check(L.osb_pcm_dev(C.c_void_p(t_e.data_ptr()), len(edges), 15.0, 1e-4, 1e-5, C.c_void_p(t_c.data_ptr()),
                                        C.c_void_p(t_c.data_ptr() + 4 * len(edges)), None, None, C.c_void_p(st)))
            for _ in range(3):
                _pcm()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                _pcm()
            e1.record(); torch.cuda.synchronize()
            widen["pcm"] = {"what": "osb_pcm_dev: 400 loop edges of one drone pair (79 800 pair checks, fp64) + maxCliqueHeu",
                            "us": e0.elapsed_time(e1) / 20 * 1e3, "clique": int(t_c[len(edges)].item()),
                            "inliers": int(sum(e["inlier"] for e in edges))}
            cases = []
            for sd in range(4):
                cs = synth.pnp_case(800 if sd == 0 else 200, 0.25, sd)
                cs.update(dict(iterations=100, thresh=0.03, seed=sd))
                cases.append(cs)
            t0p = time.perf_counter()
            outp = host.pnp_ransac(cases[:1])
            widen["pnp"] = {"what": "osb_pnp_ransac (host buffers, incl. allocation and copies): 800 correspondences, 100 hypotheses, "
                                    "LM refinement, RPerror / verify", "ms_wall": (time.perf_counter() - t0p) * 1e3,
                            "inliers": int(outp[0][1].n_inliers), "verified": int(outp[0][1].verified)}
        except Exception as e:      # noqa: BLE001
            widen["error"] = repr(e)[:200]

    # ---- BASELINE config C4 / C5 as ONE run per drone: the keyframe front-end (with the swarm exchange at N > 1) and the
    #      pose-graph back-end replayed TOGETHER -- a solver thread keeps re-solving the drone's growing sliding window (one
    #      swarm frame appended per keyframe, window = max_keyframe_num 100 frames x 5 drones, loop-5-drone.launch:15) on its
    #      own stream while the main thread processes keyframes; then the C5 keyframe step with a 50 k-row database ----
    replay = None
    if not args.no_solve:
        nd5, frames_total, window = 5, 160, 100
        gg = synth.pose_graph(nd5, frames_total, seed=11 + rank)
        fr_of = np.maximum(gg["ia"], gg["ib"]) // nd5
        order = np.argsort(fr_of, kind="stable")
        g_t, g_a, g_b, g_h, g_p, fr_s = (gg["ftype"][order], gg["ia"][order], gg["ib"][order], gg["huber"][order],
                                         gg["payload"][order], fr_of[order])
        bounds = np.searchsorted(fr_s, np.arange(frames_total + 1))
        rs = host.PoseGraphSolver(nd5 * (window + 8), 16384)
        rs.graph_clear()
        state = {"frame": 0, "dropped": 0, "solves": 0, "solve_ms": [], "stop": False, "kf": 0}

        def add_frame():                             # (only the solver thread touches the resident graph)
            f = state["frame"]
            if f >= frames_total:
                return
            off = state["dropped"] * nd5
            rs.graph_add_nodes(gg["init"][f * nd5:(f + 1) * nd5], gg["fixed"][f * nd5:(f + 1) * nd5] if state["dropped"] == 0 else None)
            a, b = bounds[f], bounds[f + 1]
            keep = (g_a[a:b] >= off) & (g_b[a:b] >= off)
            if keep.any():
                rs.graph_add_factors(g_t[a:b][keep], g_a[a:b][keep] - off, g_b[a:b][keep] - off, g_p[a:b][keep], g_h[a:b][keep])
            state["frame"] = f + 1
            if state["frame"] - state["dropped"] > window:          # sliding window (solver.cpp:186-202)
                rs.graph_drop_oldest(nd5); state["dropped"] += 1
                rs.graph_set_fixed(0, True)

        for _ in range(20):
            add_frame()

        def solver_loop():
            torch.cuda.set_device(local_rank)        # a new host thread starts on device 0
            while not state["stop"]:
                while state["frame"] < min(frames_total, 20 + state["kf"]):
                    add_frame()                      # the swarm frames that arrived since the last solve
                sm = rs.solve_resident()
                state["solves"] += 1; state["solve_ms"].append(sm.solve_ms)

        fe.finish(st); barrier()
        L.osb_set_sm_budget(148 - 16)                # the solve's cluster holds 16 SMs: keep the persistent conv grids off them
        th = threading.Thread(target=solver_loop); th.start()
        n_kf = REPLAY_KF
        t0r = time.perf_counter()
        for k in range(n_kf):
            keyframe_resident(800_000 + k)
            state["kf"] = k + 1
            if (k & 7) == 7:
                fe.finish(st)                       # keep the host at most 8 keyframes ahead, like a live stream
        fe.finish(st); barrier()
        dt = time.perf_counter() - t0r
        state["stop"] = True; th.join()
        L.osb_set_sm_budget(0)
        if world > 1:
            tt = torch.tensor([dt], device="cuda", dtype=torch.float64); dist.all_reduce(tt, op=dist.ReduceOp.MAX); dt = float(tt.item())
        replay = {"what": "C4: per drone, keyframe front-end + growing 5-drone sliding-window solve, concurrently: a solver thread "
                          "re-solves the window back to back (worst case: the reference solves at 1 Hz) while the front-end runs "
                          "with osb_set_sm_budget(132)",
                  "keyframes_per_s": world * n_kf / dt, "solves_per_s_per_drone": state["solves"] / dt,
                  "solve_ms_median": float(np.median(state["solve_ms"])) if state["solve_ms"] else None,
                  "window_frames": window, "graph_nodes": rs.graph_size()[0], "graph_factors": rs.graph_size()[1]}
        rs.close()
        # C5 keyframe step: the same step against a 50 000-row database
        fe5 = host.KeyframeFrontend(spw, comp, mean, nvw, width=W, height=H, n_dirs=N_DIRS, max_num=MAX_NUM, sp_thres=0.015,
                                    self_id=rank, db_capacity=50_000 + 2048, inner_product_thres=0.3, match_index_dist=5,
                                    zero_bottom_quarter=True, accept_min_3d_pts=10)
        for s0 in range(0, 50_000, 5000):
            fe5.db_load(synth.descriptor_db(5000, 4096, 900 + s0 + 7919 * rank), remote=False)
        rec5 = torch.zeros(lib.RECORD_BYTES, dtype=torch.uint8, device="cuda")

        def kf5(i):
            j = i % POOL
            fe5.extract(dev_up[j].data_ptr(), dev_dn[j].data_ptr(), i, rec5.data_ptr(), st, device_images=True)
            fe5.ingest_own(rec5.data_ptr(), st)
            fe5.query(rec5.data_ptr(), res_dev.data_ptr(), st)
        for i in range(5):
            kf5(i)
        fe5.finish(st); barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(60):
            kf5(100 + i)
        e1.record(); fe5.finish(st); barrier()
        ms5 = e0.elapsed_time(e1) / 60
        if world > 1:
            tt = torch.tensor([ms5], device="cuda", dtype=torch.float64); dist.all_reduce(tt, op=dist.ReduceOp.MAX); ms5 = float(tt.item())
        replay["c5_step"] = {"what": "C5 keyframe step per drone: same pipeline against a 50 000-row x 4096 f32 database (819 MB scanned per keyframe)",
                             "ms_per_keyframe": ms5, "keyframes_per_s": world * 1e3 / ms5,
                             "scan_share_gbs": 50_000 * 16384 / (ms5 - ms_keyframe + stages["db_scan"]) / 1e6 if ms5 > ms_keyframe else None}
        fe5.close()

    # ---- SURVEY 8e alternative: the 50 k-row database sharded by rows across the ranks (2 exchange steps per search) ----
    match_sharded = None
    if world > 1:
        rows = 50_000
        a, b = swarm.shard_rows(rows, rank, world)
        gen = torch.Generator(device="cuda"); gen.manual_seed(100 + rank)
        shard = torch.randn(b - a, 4096, device="cuda", generator=gen)
        shard /= shard.norm(dim=1, keepdim=True)
        rs = swarm.RowShardedIndex(shard, rows, device="cuda")
        qd = shard[0].contiguous()
        for _ in range(3):
            rs.search(qd, 10)
        torch.cuda.synchronize(); dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        e0.record()
        for _ in range(reps):
            top_s, top_i = rs.search(qd, 10)
        e1.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / reps], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        ok = int(top_i[0].item()) == a                               # my own first row is my best hit (global id)
        match_sharded = {"db_rows": rows, "rows_per_rank": b - a, "ms_per_search_round": ms,
                         "queries_per_round": world, "aggregate_gbs": rows * 16384 / ms / 1e6, "self_hit": bool(ok),
                         "note": "every rank submits one query per round: all-gather queries, scan own shard for all of "
                                 "them in one pass, all-gather candidates, merge (swarm.RowShardedIndex)"}
        rs.close(); del shard

    # ---- pose-graph solve (single GPU; replicas only) ----
    solve = None
    if not args.no_solve:
        g = synth.pose_graph_c5(0)
        solver = host.PoseGraphSolver(2048, 12288)
        solver.solve(g)                                         # warm-up
        times, walls, summ = [], [], None
        for _ in range(5):
            tw = time.perf_counter()
            poses, summ = solver.solve(g)
            walls.append((time.perf_counter() - tw) * 1e3)
            times.append(summ.solve_ms)
        lin_bytes = 12000 * (2 * 32 + 8 + 160 + 36 * 8)
        # resident graph (SURVEY 8f-4): factor list already on the device, only the initial poses are re-sent
        solver.graph_clear()
        solver.graph_add_nodes(g["init"], g["fixed"])
        solver.graph_add_factors(g["ftype"], g["ia"], g["ib"], g["payload"], g["huber"])
        solver.solve_resident()
        walls_r = []
        for _ in range(5):
            solver.graph_set_poses(0, g["init"])
            tw = time.perf_counter()
            s_res = solver.solve_resident()
            walls_r.append((time.perf_counter() - tw) * 1e3)
        resident = {"solve_wall_ms": float(np.median(walls_r)), "solve_ms": float(s_res.solve_ms),
                    "pcg_iterations": int(s_res.pcg_iterations), "final_cost": float(s_res.final_cost)}
        # config C1: the reference's default window (5 drones x 100 swarm frames, max_keyframe_num 100, loop-5-drone.launch:15)
        g1 = synth.pose_graph(5, 100, seed=0)
        solver.solve(g1)
        c1_t, c1_w = [], []
        for _ in range(5):
            tw = time.perf_counter()
            _, s1 = solver.solve(g1)
            c1_w.append((time.perf_counter() - tw) * 1e3); c1_t.append(s1.solve_ms)
        c1 = {"graph": f"C1: {g1['n_nodes']} nodes / {len(g1['ftype'])} factors", "solve_ms": float(np.median(c1_t)),
              "solve_wall_ms": float(np.median(c1_w)), "iterations": int(s1.iterations), "pcg_iterations": int(s1.pcg_iterations)}
        # "replicas only": R independent C5 windows solved CONCURRENTLY on one GPU, one 16-CTA cluster each (a solve uses
        # 16 of the 148 SMs), one handle + host thread per window -- what a ground station solving for the whole swarm does
        replicas = None
        try:
            R = 8
            solvers = [host.PoseGraphSolver(2048, 12288) for _ in range(R)]
            for sv in solvers:
                sv.graph_clear(); sv.graph_add_nodes(g["init"], g["fixed"])
                sv.graph_add_factors(g["ftype"], g["ia"], g["ib"], g["payload"], g["huber"])
                sv.solve_resident()
            reps = 6

            def work(sv):
                torch.cuda.set_device(local_rank)
                for _ in range(reps):
                    sv.graph_set_poses(0, g["init"])
                    sv.solve_resident()
            ths = [threading.Thread(target=work, args=(sv,)) for sv in solvers]
            torch.cuda.synchronize()
            tw = time.perf_counter()
            for t in ths: t.start()
            for t in ths: t.join()
            torch.cuda.synchronize()
            dt = time.perf_counter() - tw
            replicas = {"windows": R, "solves": R * reps, "solves_per_s": R * reps / dt, "ms_per_solve_amortised": dt * 1e3 / (R * reps),
                        "note": "8 resident C5 windows, one cluster of 16 CTAs each, solved concurrently from 8 host threads"}
            for sv in solvers: sv.close()
        except Exception as e:          # noqa: BLE001 -- an optional leg must not lose the bench line
            replicas = {"error": repr(e)[:200]}
        o_bj = solver.default_options(); o_bj.preconditioner = 1
        _, s_bj = solver.solve(g, o_bj)
        bj = {"solve_ms": float(s_bj.solve_ms), "pcg_iterations": int(s_bj.pcg_iterations), "iterations": int(s_bj.iterations),
              "final_cost": float(s_bj.final_cost)}
        o_64 = solver.default_options(); o_64.inner_precision = 1
        _, s_64 = solver.solve(g, o_64)
        f64 = {"solve_ms": float(s_64.solve_ms), "pcg_iterations": int(s_64.pcg_iterations), "iterations": int(s_64.iterations),
               "final_cost": float(s_64.final_cost)}
        poses, summ = solver.solve(g)                           # (phase_cycles below belong to the default solve)
        solve = {"solve_ms": float(np.median(times)),
                 "solve_wall_ms": float(np.median(walls)),   # osb_solver_solve end to end: path cover + CSR on the host, H2D of
                                                              # the factor list, kernel, D2H of the poses "iterations": int(summ.iterations),
                 "pcg_iterations": int(summ.pcg_iterations), "final_cost": float(summ.final_cost),
                 "termination": int(summ.termination), "graph": "C5: 2000 nodes / 12000 factors, Ceres-default tolerances",
                 "max_err_vs_gt_m": float(np.abs(poses[:, :3] - g["gt"][:, :3]).max()),
                 "us_per_pcg_iteration": float(np.median(times)) * 1e3 / max(1, summ.pcg_iterations),
                 "phase_cycles": solver.phase_cycles(),
                 "chain_sweep_cycles_per_iteration_by_cta_warp": (solver.chain_cycles() / max(1, summ.pcg_iterations)).round(0).tolist(),
                 "preconditioner": "chain (block-tridiagonal along the path cover, 16-node segments)",
                 "inner_precision": "fp32 PCG inside fp64 Levenberg-Marquardt",
                 "block_jacobi": bj, "fp64_inner": f64, "resident_graph": resident, "c1_window": c1, "replicas": replicas,
                 "note": "latency bound: 3 cluster barriers + 2 L2 round trips per PCG iteration; whole problem lives in shared memory / L2",
                 "approx_bytes_per_linearisation": lin_bytes}

    if rank == 0:
        line = {"metric": "keyframes/sec (SuperPoint+NetVLAD+match)", "value": value, "unit": "keyframes/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(args, world), "gpu_launches": int(launches),
                "keyframes_timed": args.steps * KF_PER_STEP, "ms_per_keyframe": ms_keyframe,
                "host_enqueue_ms_per_keyframe": host_issue_resident,
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "keyframes/s",
                        "h2d_bytes_per_step": KF_PER_STEP * 2 * N_DIRS * W * H,
                        "d2h_bytes_per_step": KF_PER_STEP * (lib.RECORD_BYTES + lib.RESULT_BYTES),
                        "ms_per_step": e2e_s * 1e3 / args.steps, "ms_per_keyframe": e2e_s * 1e3 / (args.steps * KF_PER_STEP)},
                "roofline": roofline, "roofline_conv_stack": roofline_stack, "roofline_match": roofline_match,
                "exchange": exchange, "replay_c4_c5": replay, "widen_8f": widen, "match_sweep": match_sweep, "match_sharded": match_sharded, "c2_pinhole": c2, "geometry": geometry,
                "stage_ms": stages,
                "loop_check": {"accepted": int(res.accepted), "hit_id": int(res.hit_id), "hit_score": float(res.hit_score),
                               "n_kpts": list(rec.n_kpts), "n_matches": list(res.n_matches)},
                "db_rows": int(db_rows_now), "db_rows_start": int(db_rows_start)}
        if solve:
            line["solve"] = solve
            line["solve_ms"] = solve["solve_ms"]
        if world == 1 and not args.no_trt_like:
            line["trt_like_baseline"] = trt_like_baseline(args, frames)
            line["trt_like_baseline"]["ours_e2e_over_trt_like"] = e2e_value / line["trt_like_baseline"]["value"]
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args)
        if last_step:
            dump_outputs(args.dump_outputs, *last_step)
        _emit(line)
    if world > 1:
        sw.wait(st); torch.cuda.synchronize()
        dist.barrier()
        sw.close()
        dist.destroy_process_group()


def dump_outputs(out_dir, records, results):
    """records [KF_PER_STEP, RECORD_BYTES] and results [KF_PER_STEP, RESULT_BYTES] (u8) -> out_dir/<field>.npy, one row per
    keyframe of the step: every field of osb_keyframe_record and osb_loop_result, floats as float32, integers as float64
    (exact).  List entries past their count (n_kpts per direction for the keypoint lists, n_matches / n_geo for the match
    lists) carry no result and are written as 0."""
    from omniswarm_b200 import lib
    rec = np.frombuffer(records.tobytes(), np.dtype(lib.KeyframeRecord))
    res = np.frombuffer(results.tobytes(), np.dtype(lib.LoopResult))
    cols = {name: np.array(s[name]) for s in (rec, res) for name in s.dtype.names if name != "reserved"}
    for count, names in (("n_kpts", ("local_desc", "kpts", "stereo_match", "landmarks_3d", "landmarks_flag")),
                         ("n_matches", ("match_new", "match_old")), ("n_geo", ("geo_new", "geo_old"))):
        past = np.arange(lib.MAX_KPTS)[None, None, :] >= cols[count][:, :, None]           # [keyframe, direction, entry]
        for name in names:
            cols[name][past] = 0
    os.makedirs(out_dir, exist_ok=True)
    for name, a in cols.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.dtype.kind == "f" else np.float64))


def _emit(line: dict):
    """The ONE JSON line goes to the process's original stdout; everything else that lands on fd 1 (NCCL prints its
    version banner there, libraries print progress) was redirected to stderr at start-up."""
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


if __name__ == "__main__":
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    a = parse()
    try:
        if a.impl == "reference":
            run_reference(a)
        else:
            run_ours(a)
    except BaseException:
        # fail FAST: a rank that unwinds normally here would run the CUDA teardown, which blocks for ever on streams that wait
        # for a peer's exchange stamp -- and torchrun would keep the other ranks waiting until the caller's time limit
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        os._exit(1)
