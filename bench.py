#!/usr/bin/env python
"""Benchmark of the per-frame-pair geometric core (BASELINE.json metric):

    KITTI-shape frame-pairs/sec (match + E-RANSAC + pose + LM)

Workload (config 3 of BASELINE.json): a synthetic KITTI seq-00-length run, 4541 frames x 2000
ORB-shaped keypoints (256-bit descriptors) = 4540 consecutive frame pairs per GPU.  One "step"
is one pass of the whole hot path over that sequence:
  cross-check Hamming2 matching (kitti_ba.cpp:602,641) -> findEssentialMat(RANSAC, 0.99, 1.0)
  (kitti.cpp:98-104) -> recoverPose (kitti_E.cpp:120) -> 48-point Rt Levenberg-Marquardt
  (kitti_E.cpp:170-201).
`value`  : inputs already resident in HBM, CUDA events on the library's stream.
`e2e`    : the same through the public API with HOST buffers: every step copies the sequence
           host->device from pinned memory, runs, and copies the per-pair results back.
N > 1    : one process per GPU (torchrun); every rank processes its own 4540-pair sequence
           (weak scaling, no data-path collective); the per-pair poses are all-gathered with
           NCCL inside the e2e region; times are the max over ranks.
`--impl reference`: the reference's CPU path on all host cores, bounded sample per step: the OpenCV calls the
           reference makes (cv2) + the reference's OWN Levenberg_Marquardt (oracle/_ref: jac_Rt_gen_.cpp compiled
           unmodified) when that library travelled with the snapshot, else the plain-C restatement.
Extra objects on the default line (each outside the headline timed regions):
  parity_vs_cv2   the cpu_baseline leg's cv2 results compared with the GPU results of the same pairs
  configs         the reference's other call shapes on the full 4540-pair step (kitti_E LMedS, EuRoC camera at
                  1500 kp, kitti_ba's RANSAC 0.05, ratio-mode matcher) and the 504 kitti_ba windows
  pipe_fp64       FP64-pipe fraction of the RANSAC scoring kernel against the FMA rate measured in this run
  strong_scaling  N > 1: BASELINE config 3 as written -- ONE sequence sharded by pair blocks over the ranks,
                  poses gathered (NCCL) and chained on rank 0, checked against rank 0's single-GPU run
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "KITTI-shape frame-pairs/sec (match+E-RANSAC+pose+LM)"
UNIT = "pairs/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=4541)
    ap.add_argument("--kp", type=int, default=2000)
    ap.add_argument("--method", default="ransac", choices=["ransac", "lmeds"])
    ap.add_argument("--thr", type=float, default=1.0)
    ap.add_argument("--match", default="crosscheck", choices=["crosscheck", "ratio"],
                    help="crosscheck = BFMatcher(norm, true).match (the reference, kitti_ba.cpp:602); "
                         "ratio = knnMatch(k=2) + Lowe ratio 0.8 (north_star's matcher mode)")
    ap.add_argument("--norm", default="hamming2", choices=["hamming", "hamming2"])
    ap.add_argument("--cpu-pairs", type=int, default=128, help="bounded CPU-baseline sample (pairs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="pairs", choices=["pairs", "ba_windows"],
                    help="pairs = the headline metric (default); ba_windows = BASELINE.json config 5: the 504 "
                         "kitti_ba windows of a sequence (n_zeta 10, 20 reps x 250) sharded over the GPUs (strong scaling)")
    ap.add_argument("--windows", type=int, default=504)
    ap.add_argument("--huber", type=float, default=1.0,
                    help="huber_delta of the ba_windows workload: 1.0 = the value the reference's demo tests with "
                         "(test_jac_Rt_gen.cpp:16), 1e-5 = the value jac_Rt_gen_.cpp:17 ships")
    ap.add_argument("--no-configs", action="store_true", help="skip the extra call-shape measurements (`configs`)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (rank 0) as DIR/<name>.npy "
                         "(float64), so that two builds can be compared output for output on identical inputs")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm (--impl ours)")
    return a


DUMP_MAX_ROWS = 32768           # pairs or windows dumped in full; beyond that a seeded sample (<= 42 MB either way)
DUMP_DETAIL_BYTES = 16 << 20    # matches and masks (5 x kp float64 per pair) of a seeded sample of up to 32 pairs;
                                # none when one pair's would exceed it, so a dump stays under 64 MB


def dump_rows(n, cap, rng):
    return np.arange(n) if n <= cap else np.sort(rng.choice(n, cap, replace=False))


def dump_arrays(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(v, dtype=np.float64))


def dump_pairs(out_dir, pipe, P, kp):
    """What a caller of the resident path receives after its last step: the per-pair results (epivo_seq_download),
    one array per field, and the matches and masks (epivo_seq_get_matches / _masks) of a seeded sample of pairs,
    padded with -1 to kp entries.  pair_index / detail_pair_index name the pairs dumped."""
    res = pipe.download(0, P)
    rng = np.random.default_rng(0)
    rows = dump_rows(P, DUMP_MAX_ROWS, rng)
    out = {"pair_index": rows}
    out.update({f: res[f][rows] for f in res.dtype.names})
    detail = dump_rows(P, min(32, DUMP_DETAIL_BYTES // (40 * kp)), rng)
    cols = {k: np.full((len(detail), kp), -1.0) for k in ("match_query", "match_train", "match_distance",
                                                          "essential_mask", "pose_mask")}
    for j, i in enumerate(detail):
        qi, ti, d = pipe.matches(int(i))
        em, pm = pipe.masks(int(i))
        for k, v in zip(cols, (qi, ti, d, em, pm)):
            cols[k][j, :len(v)] = v
    out["detail_pair_index"] = detail
    out.update(cols)
    dump_arrays(out_dir, out)


def config_of(a, world):
    """The `config` object: identical keys and values in both arms (the driver compares them)."""
    P = a.frames - 1
    return {"workload": workload_name(a), "pairs_per_gpu": P,
            "l2": "inputs (%d MB/GPU) larger than L2" % round((a.frames * a.kp * 40) / 1e6),
            "parallelism": f"pairs sharded, {world} x 1 GPU, no data-path collective"}


def workload_name(a):
    return (f"kitti_E synthetic seq-00-length run: {a.frames} frames x {a.kp} kp x 256-bit descriptors, "
            f"{a.frames - 1} pairs per GPU; BFMatcher({a.norm.upper()}, "
            f"{'crossCheck' if a.match == 'crosscheck' else 'knnMatch k=2 + ratio 0.8'}) + findEssentialMat("
            f"{a.method.upper()}, 0.99, {a.thr}) + recoverPose + 48-pt LM")


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "200", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.25)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 8]
        os.unlink(self.f.name)
        if not rows:
            return out
        sm = [float(r[1]) for r in rows if r[1].strip().replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if r[2].strip().replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = set()
        for r in rows:
            for k, nm in enumerate(names):
                if r[5 + k].strip().lower() == "active":
                    reasons.add(nm)
        out.update(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                   reasons=sorted(reasons), samples=len(rows))
        return out


def bind_near_gpu(local):
    """N > 1: run this rank (and first-touch its pinned staging buffers) on the host cores NVML reports as local
    to its GPU, so that eight ranks pulling 363 MB per step do not all cross the socket interconnect.
    Best effort: any failure leaves the affinity as it was."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(local)
        bus = "%08X:%02X:%02X.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        ncpu = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [i for i in range(ncpu) if (mask[i // 64] >> (i % 64)) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if cpus and len(cpus) < len(allowed):
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


def make_inputs(a, rank):
    from epivo_b200 import synth
    seq = synth.make_sequence(a.frames, a.kp, seed=synth.seed_for(3, rank))
    return seq


def run_reference(a):
    """`--impl reference`: rank 0 only; bounded sample per step on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from epivo_b200 import synth
    from oracle import cpu_reference as R
    per_step = max(8, min(a.cpu_pairs, a.frames - 1))
    seq = synth.make_sequence(min(a.frames, per_step + 1), a.kp, seed=synth.seed_for(3, 0))
    method = 8 if a.method == "ransac" else 4
    cores = os.cpu_count() or 1
    pool = R.CpuPool(seq.kps, seq.descs, seq.K, method, 0.99, a.thr, cores=cores,
                     norm=7 if a.norm == "hamming2" else 6, ratio=None if a.match == "crosscheck" else 0.8)
    idx = list(range(seq.n_pairs))
    for _ in range(a.warmup):
        pool.run(idx[:max(cores, 8)])
    t0 = time.perf_counter()
    for _ in range(a.steps):
        pool.run(idx)
    dt = time.perf_counter() - t0
    pool.close()
    value = a.steps * len(idx) / dt
    kind = "reference" if (R.HAVE_CV2 and R.lm_kind() == "reference") else "port"
    sample = (f"{len(idx)} pairs per step of the same synthetic sequence; " + R.describe()
              + f"; {cores} worker processes x 1 thread, pair-parallel")
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8+f64", "data": "synthetic", "impl": "reference",
            "config": config_of(a, max(a.gpus, 1)),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


_REAL_STDOUT = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version line when
    NCCL_DEBUG is set on the box), so fd 1 is pointed at stderr for the whole run and the JSON line goes to the
    saved original descriptor."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def windows_measure(a, ctx, world, rank, local, dist, steps, warmup, windows=None):
    """BASELINE.json config 5: the windows of one sequence (n_zeta 10, reps {(i,i),(0,i)} x 250 correspondences,
    test_jac_Rt_gen.cpp:282-297), sharded over the ranks in contiguous blocks (strong scaling: the total is fixed),
    one batched Levenberg_Marquardt launch per rank.  -> dict(kernel ms, wall ms, launches, ...), max over ranks."""
    import torch
    from epivo_b200 import api, shard, synth
    windows = a.windows if windows is None else windows
    nz, N = 10, 250
    reps = [(i, i) for i in range(nz)] + [(0, i) for i in range(nz)]
    lo, hi = shard.shard_range(windows, world, rank)
    B = hi - lo
    data = [synth.gen_scene_sequence(500 + (lo + b) % 64, N, nz, reps) for b in range(min(B, 64))]

    def pinned(k):
        t = torch.from_numpy(np.stack([data[b % len(data)][k] for b in range(B)])).pin_memory()
        return t, t.numpy()
    keep = [pinned(k) for k in (1, 2, 3)]
    T0, pr, p_r = (x[1] for x in keep)
    w = [1.0] * len(reps)

    def step():
        return api.Levenberg_Marquardt_batch(nz, 1e-8, reps, w, 1e-2, T0, pr, p_r, huber_delta=a.huber, ctx=ctx)
    for _ in range(max(warmup, 1)):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    n0 = ctx.launch_count
    t0 = time.perf_counter()
    k_ms = 0.0
    for _ in range(steps):
        T, res, its = step()
        k_ms += ctx.last_kernel_ms()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3 / steps
    k_ms /= steps
    launches = ctx.launch_count - n0
    if world > 1:
        t = torch.tensor([k_ms, wall_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        k_ms, wall_ms = float(t[0].item()), float(t[1].item())
        dist.barrier()
    return {"windows": windows, "B": B, "k_ms": k_ms, "wall_ms": wall_ms, "launches": int(launches),
            "mean_iters": float(its.mean()) if B else 0.0, "h2d": int(T0.nbytes + pr.nbytes + p_r.nbytes),
            "d2h": int(T0.nbytes + B * 28), "data": data, "nz": nz, "reps": reps,
            "outputs": {"T": T, "H_norm_r_norm_lambda": res, "iters": its}}


def run_windows(a):
    """`--workload ba_windows` (not the headline line): value = windows / max over ranks of the kernel time; e2e = the
    same through epivo_lm_rt_batch with pinned host buffers (H2D of the reprojections + D2H of the refined chains)."""
    import torch
    import torch.distributed as dist
    from epivo_b200 import api
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = api.Context(local)
    clocks = ClockSampler(local)
    m = windows_measure(a, ctx, world, rank, local, dist, a.steps, a.warmup)
    clk = clocks.stop()
    if a.dump_outputs and rank == 0:
        rows = dump_rows(m["B"], DUMP_MAX_ROWS, np.random.default_rng(0))
        dump_arrays(a.dump_outputs, {"window_index": rows, **{k: v[rows] for k, v in m["outputs"].items()}})
    line = {"metric": "kitti_ba windows/sec (windowed Rt LM, n_zeta 10, 20 reps x 250 correspondences, 30 iterations, "
                      "huber_delta %g)" % a.huber,
            "value": a.windows / (m["k_ms"] * 1e-3), "unit": "windows/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": m["k_ms"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": f"BASELINE config 5: {a.windows} windows (sequence.hpp scenes), contiguous blocks per rank, "
                                   f"{m['B']} on rank {rank}; huber_delta {a.huber:g} (jac_Rt_gen_.cpp:17 ships 1e-5, "
                                   f"test_jac_Rt_gen.cpp:16 tests 1.0)",
                       "parallelism": f"windows sharded, {world} x 1 GPU, no collective"},
            "clocks": clk,
            "e2e": {"value": a.windows / (m["wall_ms"] * 1e-3), "unit": "windows/s", "ms_per_step": m["wall_ms"],
                    "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": m["d2h"]},
            "gpu_launches": m["launches"], "mean_iters": m["mean_iters"]}
    if world == 1 and not a.no_cpu_baseline:
        line["cpu_baseline"] = windows_cpu_baseline(a, m)
    if rank == 0:
        emit(line)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def windows_cpu_baseline(a, m):
    from oracle import cpu_reference as R
    cores = os.cpu_count() or 1
    n = 2 * cores
    v = R.windows_rate(m["data"], m["nz"], m["reps"], n, cores=cores, huber_delta=a.huber)
    return {"value": v, "unit": "windows/s", "cores": cores, "kind": "port",
            "sample": f"{n} windows of the same shape; plain-C restatement of the reference LM (pinned to the reference's "
                      f"own build, tests/test_oracle_ref.py; that build -- g++ -O0 against a stand-in Eigen -- is ~100x "
                      f"slower and would flatter the ratio), {cores} processes x 1 thread"}


class PairsRunner:
    """One resident sequence + pinned host copies; measures a parameter set both device-resident and end to end."""

    def __init__(self, ctx, seq, local, world, dist):
        import torch
        from epivo_b200 import api
        self.torch, self.api, self.ctx, self.seq, self.world, self.dist = torch, api, ctx, seq, world, dist
        self.F, self.P, self.kp = seq.n_frames, seq.n_pairs, seq.kps.shape[1]
        self.h_kps = torch.from_numpy(seq.kps).pin_memory()          # torch owns the pinned allocation;
        self.h_desc = torch.from_numpy(seq.descs).pin_memory()       # numpy views go to the C ABI
        self.kps_np, self.desc_np = self.h_kps.numpy(), self.h_desc.numpy()
        self.pipe = api.SequencePipeline(self.F, self.kp, ctx=ctx)
        self.stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local))
        self.h_res = torch.zeros(self.P * api.RESULT_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
        self.results = self.h_res.numpy().view(api.RESULT_DTYPE)
        if world > 1:                                                # staging of the pose gather: allocated once
            self.T_pin = torch.zeros((self.P, 4, 4), dtype=torch.float64).pin_memory()
            self.T_pin_np = self.T_pin.numpy()
            self.T_dev = torch.empty((self.P, 4, 4), dtype=torch.float64, device="cuda")
            self.T_all = torch.empty((world * self.P, 4, 4), dtype=torch.float64, device="cuda")
        self.pipe.upload(self.kps_np, self.desc_np)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([float(x)], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def resident(self, prm, steps, warmup):
        """EXACTLY `steps` steps with the inputs resident in HBM; CUDA events on the library's stream."""
        torch, pipe, P = self.torch, self.pipe, self.P
        for _ in range(warmup):
            pipe.run(prm, 0, P)
        self.ctx.sync()
        launches0 = self.ctx.launch_count
        stage_acc = np.zeros(16, dtype=np.float64)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(steps):
            pipe.run(prm, 0, P)
            stage_acc += pipe.stage_ms()      # syncs the stream (microseconds against a >= 17 ms step)
        e1.record(self.stream)
        self.barrier()
        ms_step = self.max_over_ranks(e0.elapsed_time(e1) / steps)
        return ms_step, stage_acc / steps, self.ctx.launch_count - launches0

    def end_to_end(self, prm, steps, warmup=2, gather=True):
        """The same through the public API with HOST buffers: H2D of the sequence (pipelined under the matcher),
        run, D2H of the per-pair results, and -- N > 1 -- the NCCL all-gather of the poses, every step."""
        torch, pipe, world = self.torch, self.pipe, self.world
        for _ in range(warmup):
            pipe.process(prm, self.kps_np, self.desc_np, self.results)
        self.barrier()
        t0 = time.perf_counter()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record(self.stream)
        t_proc = 0.0
        for _ in range(steps):
            tp = time.perf_counter()
            pipe.process(prm, self.kps_np, self.desc_np, self.results)
            t_proc += time.perf_counter() - tp
            if world > 1 and gather:          # the only collective: per-pair poses -> every rank (NCCL)
                np.copyto(self.T_pin_np, self.results["T"])                  # results are pinned: strided field -> pinned 4x4s
                self.T_dev.copy_(self.T_pin, non_blocking=True)
                self.dist.all_gather_into_tensor(self.T_all, self.T_dev)
        e3.record(self.stream)
        self.barrier()
        wall = time.perf_counter() - t0
        ms = max(e2.elapsed_time(e3), wall * 1e3) / steps          # host-side staging counts too
        self.process_ms_per_rank = None                            # this rank's own epivo_seq_process time, all ranks
        if world > 1:
            t = torch.tensor([t_proc * 1e3 / steps], device="cuda", dtype=torch.float64)
            allt = [torch.empty_like(t) for _ in range(world)]
            self.dist.all_gather(allt, t)
            self.process_ms_per_rank = [round(float(x.item()), 3) for x in allt]
        return self.max_over_ranks(ms)

    def close(self):
        self.pipe.close()


def front_end_measure(ctx, frames=128):
    """N4: FastFeatureDetector(40) on every frame and calcOpticalFlowPyrLK into the next one (kitti_E.cpp:70-84) for a
    KITTI-sized synthetic sequence, through the host API (the frames are uploaded inside the timed region)."""
    from epivo_b200 import api
    rng = np.random.default_rng(12)
    tex = rng.integers(0, 256, (376 + 64, 1241 + 64)).astype(np.float32)
    for _ in range(4):                                    # smooth texture: four 3 x 3 box filters (~3000 FAST-40 corners, KITTI-like)
        tex = sum(np.roll(np.roll(tex, dy, 0), dx, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1)) / 9.0
    tex = ((tex - tex.min()) / (tex.max() - tex.min()) * 255).astype(np.uint8)
    seq = np.stack([tex[32 + (k % 5):32 + (k % 5) + 376, 32 + 2 * (k % 7):32 + 2 * (k % 7) + 1241] for k in range(frames)])
    from epivo_b200 import synth
    K = synth.KITTI_K.astype(np.float32)                                 # the KITTI camera of kitti_E.cpp:38-40
    prm = api.default_params(K, method=api.LMEDS, prob=0.99, threshold=0.01)   # kitti_E.cpp:98-104
    best, pipe = None, None
    for _ in range(3):
        t0 = time.perf_counter()
        det = api.fastDetect(seq[:-1], 40, True, max_keypoints=8192, ctx=ctx)
        t1 = time.perf_counter()
        nxt, st = api.trackSequenceLK(seq, [d[0] for d in det], ctx=ctx)
        t2 = time.perf_counter()
        p0 = [det[i][0][st[i] == 1] for i in range(frames - 1)]          # kitti_E.cpp:86-95
        p1 = [nxt[i][st[i] == 1] for i in range(frames - 1)]
        if pipe is None:
            pipe = api.SequencePipeline(frames, max(8, max(len(p) for p in p0)), ctx=ctx)
        res = pipe.process_points(prm, p0, p1)
        t3 = time.perf_counter()
        if best is None or t3 - t0 < best[0]:
            best = (t3 - t0, t1 - t0, t2 - t1, t3 - t2)
    pipe.close()
    n = frames - 1
    return {"workload": "the loop body of kitti_E.cpp:54-201 from %d synthetic 1241x376 frames: FAST-9/16 threshold 40 with "
                        "suppression, 21x21 pyramidal LK (3 levels, 30 iterations) of every corner into the next frame, then "
                        "findEssentialMat(LMEDS, .99, .01) + recoverPose + 48-pt LM on the tracks" % frames,
            "value": n / best[0], "unit": "frames/s", "fast_ms_per_frame": best[1] * 1e3 / n, "lk_ms_per_pair": best[2] * 1e3 / n,
            "geometry_ms_per_pair": best[3] * 1e3 / n,
            "mean_corners": float(np.mean([len(d[0]) for d in det])), "tracked_frac": float(np.mean([s.mean() for s in st])),
            "mean_inlier_frac": float(np.mean(res["n_inliers"] / np.maximum(res["n_matches"], 1))),
            "includes": "host->device upload of the frames / tracks and device->host of the points / results, host-side "
                        "status filtering, wall clock"}


def orb_front_end_measure(ctx, frames=32, batch=8, cpu=True):
    """N4: kitti_ba's front end (extract_good_kp, kitti_ba.cpp:114-156, then really_robust_ass's matcher, :602,641) from
    KITTI-sized synthetic frames through the host API: ORB(10000, 1.2, 8, 15, 0, 2, FAST_SCORE) detect + compute on every
    frame, then BFMatcher(HAMMING2, crossCheck) at ~10000 x 10000 + findEssentialMat(RANSAC, .99, .05) + recoverPose + LM
    on consecutive frames."""
    from epivo_b200 import api, synth
    big = synth.corner_scene(376 + 40, 1241 + 3 * frames + 8, 31)
    seq = np.stack([big[(k % 5):(k % 5) + 376, 3 * k:3 * k + 1241] for k in range(frames)])
    K = synth.KITTI_K.astype(np.float32)
    prm = api.default_params(K, method=api.RANSAC, prob=0.99, threshold=0.05)          # kitti_ba.cpp:308
    cap = 12288
    pipe = api.SequencePipeline(frames, cap, ctx=ctx)
    best, host, same = None, None, True
    for _ in range(3):
        # (a) ORB through its own host-buffer call (what the drop-in epivo::ORB does), packed and uploaded by the host
        t0 = time.perf_counter()
        feats = []
        for i in range(0, frames, batch):
            feats += api.orbDetectAndCompute(seq[i:i + batch], 10000, max_keypoints=cap, ctx=ctx)
        t1 = time.perf_counter()
        counts = np.array([len(k) for k, _ in feats], dtype=np.int32)
        kps = np.zeros((frames, cap, 2), dtype=np.float32)
        descs = np.zeros((frames, cap, 32), dtype=np.uint8)
        for i, (k, d) in enumerate(feats):                                             # KeyPoint::convert, kitti_ba.cpp:145
            kps[i, :counts[i], 0], kps[i, :counts[i], 1] = k["x"], k["y"]
            descs[i, :counts[i]] = d
        pipe.upload(kps, descs)
        pipe.set_counts(counts)
        pipe.run(prm, 0, frames - 1)
        res_host = pipe.download(0, frames - 1).copy()
        t2 = time.perf_counter()
        if host is None or t2 - t0 < host[0]:
            host = (t2 - t0, t1 - t0, t2 - t1)
        # (b) frames -> ORB -> frame slots on the device (epivo_seq_extract_orb), then the same pair pipeline
        t0 = time.perf_counter()
        for i in range(0, frames, batch):
            pipe.extract_orb(seq[i:i + batch], i, 10000)
        t1 = time.perf_counter()
        pipe.run(prm, 0, frames - 1)
        res = pipe.download(0, frames - 1)
        t2 = time.perf_counter()
        same = same and res.tobytes() == res_host.tobytes()                            # the two routes agree byte for byte
        if best is None or t2 - t0 < best[0]:
            best = (t2 - t0, t1 - t0, t2 - t1)
    pipe.close()
    cpu_ref = None
    if cpu:                                # the same OpenCV calls on the host cores, a few frames (not oracle code: cv2 itself)
        try:
            import cv2
            orb = cv2.ORB_create(10000, 1.2, 8, 15, 0, 2, cv2.ORB_FAST_SCORE)
            m = min(frames, 6)
            t0 = time.perf_counter()
            for i in range(m):
                kp = orb.detect(seq[i], None)
                kp, d = orb.compute(seq[i], kp)
            cpu_ref = {"value": (time.perf_counter() - t0) * 1e3 / m, "unit": "ms per frame", "what": "cv2 %s ORB detect + compute, "
                       "OpenCV's own threading (%d host cores)" % (cv2.__version__, os.cpu_count() or 1),
                       "identical_to_gpu_last_frame": bool(len(kp) == len(feats[m - 1][0]) and np.array_equal(d, feats[m - 1][1]))}
        except Exception as e:             # noqa: BLE001 -- cv2 missing or failing must not cost the GPU numbers
            cpu_ref = {"error": "%s: %s" % (type(e).__name__, e)}
    return {"workload": "kitti_ba.cpp:114-156 + :602,641 from %d synthetic 1241x376 frames: ORB::create(10000, 1.2f, 8, 15, 0, 2, "
                        "FAST_SCORE) detect + compute (batches of %d frames), BFMatcher(NORM_HAMMING2, crossCheck) on consecutive "
                        "frames, findEssentialMat(RANSAC, .99, .05) + recoverPose + 48-pt LM" % (frames, batch),
            "value": frames / best[0], "unit": "frames/s", "orb_ms_per_frame": best[1] * 1e3 / frames,
            "match_geometry_ms_per_pair": best[2] * 1e3 / (frames - 1), "mean_keypoints": float(counts.mean()),
            "via_host_buffers": {"value": frames / host[0], "unit": "frames/s", "orb_ms_per_frame": host[1] * 1e3 / frames,
                                 "pack_upload_match_geometry_ms_per_pair": host[2] * 1e3 / (frames - 1),
                                 "note": "epivo_orb_detect_and_compute -> host -> epivo_seq_upload", "results_identical": bool(same)},
            "mean_matches": float(res["n_matches"].mean()), "mean_inlier_frac": float(np.mean(res["n_inliers"] / np.maximum(res["n_matches"], 1))),
            "cv2_orb": cpu_ref,
            "includes": "host->device upload of the frames, ORB into the frame slots on the device (epivo_seq_extract_orb), "
                        "matcher + geometry, device->host of the results, wall clock"}


def rot_angle(a, b):
    return float(np.arccos(np.clip((np.trace(a.T @ b) - 1) / 2, -1, 1)))


def strong_scaling_leg(a, ctx, local, world, rank, dist, prm, runner0):
    """BASELINE config 3 as written: ONE 4541-frame sequence (rank 0's), pairs sharded in contiguous blocks
    (shard.shard_range, halo of one frame), every rank runs its block from host buffers, the per-pair poses are
    all-gathered (NCCL) into sequence order and rank 0 chains them (kitti_E.cpp:218-228).  Checked against rank 0's
    own single-GPU run of all pairs."""
    import torch
    from epivo_b200 import api, shard, synth
    seq0 = runner0.seq if rank == 0 else synth.make_sequence(a.frames, a.kp, seed=synth.seed_for(3, 0))
    P = seq0.n_pairs
    lo, hi = shard.shard_range(P, world, rank)
    f0, f1 = shard.frames_for(lo, hi)
    nb = hi - lo
    h_kps = torch.from_numpy(np.ascontiguousarray(seq0.kps[f0:f1])).pin_memory()
    h_desc = torch.from_numpy(np.ascontiguousarray(seq0.descs[f0:f1])).pin_memory()
    pipe = api.SequencePipeline(max(f1 - f0, 2), a.kp, ctx=ctx)
    h_res = torch.zeros(max(nb, 1) * api.RESULT_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
    res = h_res.numpy().view(api.RESULT_DTYPE)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local))

    def step():
        if nb > 0:
            pipe.process(prm, h_kps.numpy(), h_desc.numpy(), res)
        allT = shard.gather_poses(np.ascontiguousarray(res["T"][:nb]), P, world, rank, dist=dist, device="cuda")
        return api.chain_poses(allT, ctx=ctx) if rank == 0 else None, allT      # device block scan (cloud.cu)
    for _ in range(2):
        step()
    dist.barrier()
    torch.cuda.synchronize()
    steps = 3
    t0 = time.perf_counter()
    for _ in range(steps):
        poses, allT = step()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / steps
    t = torch.tensor([ms], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    out = {"pairs": P, "ms_per_step": ms, "value": P / (ms * 1e-3), "unit": UNIT, "scaling": "strong",
           "pairs_on_rank0": nb, "includes": "H2D of the rank's frames + run + D2H + NCCL all-gather of the poses + pose chain on "
                                            "rank 0's GPU (epivo_chain_poses), wall clock, max over ranks"}
    if rank == 0:
        single = runner0.pipe.process(prm, runner0.kps_np, runner0.desc_np, runner0.results)
        Ts = np.array(single["T"])
        out["equal_to_single_gpu"] = bool(np.array_equal(Ts, allT))
        out["max_abs_diff_vs_single_gpu"] = float(np.abs(Ts - allT).max())
        out["chain_max_abs_diff"] = float(np.nanmax(np.abs(poses - api.chain_poses(Ts, ctx=ctx))))
        out["chain_vs_host_restatement"] = float(np.nanmax(np.abs(poses - shard.chain_poses(Ts))))
    pipe.close()
    return out


def main():
    a = parse()
    quiet_stdout()
    if a.impl == "reference":
        run_reference(a)
        return
    if a.workload == "ba_windows":
        run_windows(a)
        return
    import torch
    import torch.distributed as dist
    from epivo_b200 import api, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    near_cpus = bind_near_gpu(local) if world > 1 else 0
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    seq = make_inputs(a, rank)
    ctx = api.Context(local)
    run = PairsRunner(ctx, seq, local, world, dist)
    P, kp = run.P, a.kp
    method = api.RANSAC if a.method == "ransac" else api.LMEDS
    Kf = seq.K.astype(np.float32)
    prm = api.default_params(Kf, method=method, threshold=a.thr,
                             match_mode=1 if a.match == "crosscheck" else 2, ratio=0.8,
                             norm=api.NORM_HAMMING2 if a.norm == "hamming2" else api.NORM_HAMMING)

    # ---------------- headline: device-resident, then end to end with host buffers ------------------
    clocks = ClockSampler(local)
    ms_step, stages, launches = run.resident(prm, a.steps, a.warmup)
    if a.dump_outputs and rank == 0:
        dump_pairs(a.dump_outputs, run.pipe, P, kp)
    value = world * P / (ms_step * 1e-3)
    ms_e2e = run.end_to_end(prm, a.steps)
    e2e_value = world * P / (ms_e2e * 1e-3)
    clk = clocks.stop()
    results = run.results.copy()

    # ---------------- roofline of the dominant kernel (the matcher) -------------------------
    ms_match = stages[7]                                     # tile kernel alone, summed over chunk launches
    n_chunk_launches = int(round(stages[8]))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback"
    # algorithmic bytes per pair (SURVEY 8d): 32*(nq+nt) descriptor bytes in + 16*nq key/match bytes out
    bytes_per_pair = 32 * (kp + kp) + 16 * kp
    achieved_gbs = bytes_per_pair * P / (ms_match * 1e-3) / 1e9
    popc_peak = ctx.microbench(0)                            # POPC.32 thread-ops/s, measured now on this GPU
    lop_peak = ctx.microbench(4)
    fp64_peak = ctx.microbench(2)                            # FP64 FMA thread-ops/s
    # algorithmic POPC.32 per pair: nq*nt*(256/32) for plain Hamming; the Hamming2 bit-plane form
    # needs nq*nt*4 -- report against the instruction count the kernel actually needs (4)
    popc_per_pair = kp * kp * (4 if a.norm == "hamming2" else 8)
    achieved_popc = popc_per_pair * P / (ms_match * 1e-3)
    # DRAM traffic of one matcher launch over the default workload: NOT measured in this run (it needs ncu); the figure
    # is dram__bytes_read.sum + dram__bytes_write.sum of the `ncu --set full` capture named in traffic_source.  It is
    # BELOW the algorithmic bytes because consecutive pairs share a frame (train set of pair i = query set of pair
    # i+1) that is still in L2.  Only valid for the profiled shape.
    default_shape = (a.frames == 4541 and a.kp == 2000 and n_chunk_launches == 1 and a.norm == "hamming2"
                     and a.match == "crosscheck")
    roofline = {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved_gbs / hbm_peak, "traffic": 386.8e6 if default_shape else None,
                "traffic_source": "profiles/r1_ncu_full_top_kernels.csv (ncu --set full of this command, not measured live)"
                                  if default_shape else None,
                "peak_source": peak_src,
                "kernel": "match_tile_kernel<8,%s%s>" % (a.norm.upper(), ",TOP2" if a.match == "ratio" else ""), "launches_per_step": n_chunk_launches,
                "algorithmic_bytes_per_launch": bytes_per_pair * P / max(n_chunk_launches, 1),
                "ms_per_step_in_kernel": ms_match,
                "note": "the matcher is bound by the integer pipes (POPC on XU, LOP3 on ALU), not HBM "
                        "(AI ~ 100 popc/byte, so the HBM fraction is < 1 % by construction): see pipe"}
    # POPC instructions the kernel ISSUES per descriptor pair: carry-save compression counts 4 (Hamming2 planes)
    # or 8 (plain Hamming) algorithmic words with 3 or 4 POPC
    issued_per_alg = (3.0 / 4.0) if a.norm == "hamming2" else (4.0 / 8.0)
    issued_popc = achieved_popc * issued_per_alg
    pipe_roof = {"bound": "popc32 (XU pipe) / LOP3 (ALU pipe)", "achieved": issued_popc / 1e9,
                 "peak": popc_peak / 1e9, "unit": "Gpopc/s (issued)", "frac": issued_popc / popc_peak,
                 "algorithmic_Gpopc_s": achieved_popc / 1e9, "algorithmic_frac": achieved_popc / popc_peak,
                 "alu_peak_Gops": lop_peak / 1e9,
                 "work": "nq*nt*%d POPC.32 per pair (%s), one direction + fused column minima" % (
                     (4, "Hamming2 on bit planes") if a.norm == "hamming2" else (8, "plain Hamming")),
                 "note": "frac = issued POPC.32 rate / POPC.32 peak measured in this run (epivo_microbench); the "
                         "algorithmic rate is higher because carry-save adders compress the words before counting; "
                         "ncu (profiles/): XU (POPC) pipe 88 %, ALU (LOP3) pipe 89 % of peak"}

    def fp64_block(res, st):
        """FP64 pipe of the RANSAC / LMedS scoring: (models scored) x (correspondences) Sampson tests at 17 FP64
        instructions each (fused pre-filter path, DESIGN K3) over the time of the essential rounds (essential stage
        minus sampling + minimal solver), against the FP64 FMA rate measured in this run."""
        evals = float((res["n_models"].astype(np.float64) * res["n_matches"]).sum())
        ms_rounds = max(st[3] - st[2], 1e-6)
        ach = 17.0 * evals / (ms_rounds * 1e-3)
        return {"kernel": "ess_round_kernel (+ bookkeeping inside the essential rounds)", "bound": "fp64 pipe",
                "achieved": ach / 1e9, "peak": fp64_peak / 1e9, "unit": "G FP64 instr/s", "frac": ach / fp64_peak,
                "model_x_point_tests_per_step": evals, "ms_per_step_in_rounds": ms_rounds,
                "fp64_instr_per_test": 17}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32-popc+f64", "data": "synthetic",
            "config": config_of(a, world),
            "host_affinity": (f"rank bound to {near_cpus} GPU-local cores (NVML)" if near_cpus else "unchanged"),
            "clocks": clk,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(run.kps_np.nbytes + run.desc_np.nbytes),
                    "d2h_bytes_per_step": int(run.results.nbytes), "ms_per_step": ms_e2e},
            "gpu_launches": int(launches),
            "roofline": roofline, "pipe": pipe_roof, "pipe_fp64": fp64_block(results, stages),
            "stages_ms_per_step": {k: float(stages[i]) for i, k in
                                   enumerate(["total", "match", "presolve", "essential", "pose", "lm", "finish",
                                              "match_kernel"])},
            "quality": {"mean_matches": float(results["n_matches"].mean()),
                        "mean_inliers": float(results["n_inliers"].mean()),
                        "mean_good": float(results["n_good"].mean()),
                        "mean_ransac_iters": float(results["ransac_iters"].mean()),
                        "lm_ran_frac": float(results["lm_ran"].mean()),
                        "lm_reverted_frac": float(results["lm_reverted"].mean()),   # kitti_E.cpp:198-200 reverts when r_norm > 1e-9
                        "median_rot_err_rad": float(np.median([rot_angle(results["R"][i], seq.R[i])
                                                               for i in range(0, P, max(1, P // 256))]))}}
    if world > 1:
        # copy-only ceiling of this box class (tools/h2d_ceiling.py, all ranks copying 363 MB at once, committed under
        # profiles/): an e2e step cannot end before its input has landed
        ceil_ms = {2: 6.56, 4: 12.65, 8: 15.60}.get(world)
        e2e_lim = {"aggregate_h2d_GBps": world * (run.kps_np.nbytes + run.desc_np.nbytes) / (ms_e2e * 1e-3) / 1e9,
                   "h2d_copy_only_ms_per_step": ceil_ms,
                   "h2d_copy_only_source": "profiles/r2_h2d_ceiling_%dgpu.json (measured on this pool, not in this run)" % world
                   if ceil_ms else None}
        line["e2e"]["limiter"] = ("host->device input path: %d ranks x %.0f MB per step = %.0f GB/s aggregate through the host; "
                                  "the step ends one matcher piece + the geometry after the last byte lands"
                                  % (world, (run.kps_np.nbytes + run.desc_np.nbytes) / 1e6, e2e_lim["aggregate_h2d_GBps"]))
        line["e2e"].update(e2e_lim)
        line["e2e"]["process_ms_per_rank"] = run.process_ms_per_rank     # the slowest rank sets the step (one gather per step)

    # ---------------- the reference's other call shapes, full step each (not the headline) ---------------
    if not a.no_configs:
        cfgs = {}

        def shape(name, r, p, note, steps=3):
            ms_r, st, _ = r.resident(p, steps, 1)
            ms_e = r.end_to_end(p, 2, warmup=1, gather=False)
            res = r.results
            cfgs[name] = {"workload": note, "value": world * r.P / (ms_r * 1e-3), "unit": UNIT, "ms_per_step": ms_r,
                          "e2e": world * r.P / (ms_e * 1e-3), "e2e_ms_per_step": ms_e,
                          "mean_ransac_iters": float(res["ransac_iters"].mean()), "mean_inliers": float(res["n_inliers"].mean()),
                          "stages_ms": {"match": float(st[1]), "presolve": float(st[2]), "essential": float(st[3]),
                                        "pose": float(st[4]), "lm": float(st[5])},
                          "pipe_fp64": fp64_block(res.copy(), st)}
        shape("kitti_E LMEDS(.99,.01)", run, api.default_params(Kf, method=api.LMEDS, prob=0.99, threshold=0.01),
              "kitti_E.cpp:98-104 on the headline sequence")
        shape("kitti_ba RANSAC(.99,.05)", run, api.default_params(Kf, method=api.RANSAC, prob=0.99, threshold=0.05),
              "kitti_ba.cpp:308 (1000 iterations per pair) on the headline sequence", steps=2)
        shape("ratio-mode matcher", run, api.default_params(Kf, method=method, threshold=a.thr, match_mode=2, ratio=0.8,
                                                            norm=api.NORM_HAMMING),
              "knnMatch(k=2) + Lowe ratio 0.8 on plain 256-bit Hamming (north_star's matcher mode), then the headline geometry")
        seq_e = synth.make_sequence(a.frames, 1500, seed=synth.seed_for(2, rank), K=synth.EUROC_K, size=synth.EUROC_SIZE,
                                    depth=(1.0, 8.0), px_sigma=0.3, outlier_frac=0.25, step=(0.03, 0.07))
        run_e = PairsRunner(ctx, seq_e, local, world, dist)
        shape("euroc_E RANSAC(.99,.3) 1500 kp", run_e,
              api.default_params(synth.EUROC_K.astype(np.float32), method=api.RANSAC, prob=0.99, threshold=0.3,
                                 fallback_t=(0.0, 0.0, 1.0)),
              "euroc_E.cpp:202-208: EuRoC camera, 752x480, %d frames x 1500 kp" % a.frames)
        run_e.close()
        del run_e, seq_e
        m = windows_measure(a, ctx, world, rank, local, dist, 3, 1)
        cfgs["kitti_ba windows"] = {"workload": "BASELINE config 5: %d windows (n_zeta 10, 20 reps x 250), sharded over the ranks "
                                                "(strong scaling), huber_delta %g" % (m["windows"], a.huber),
                                    "value": m["windows"] / (m["k_ms"] * 1e-3), "unit": "windows/s", "ms_per_step": m["k_ms"],
                                    "e2e": m["windows"] / (m["wall_ms"] * 1e-3), "e2e_ms_per_step": m["wall_ms"],
                                    "mean_iters": m["mean_iters"], "windows_on_rank0": m["B"]}
        for name, fn in (("kitti_E from frames: FAST(40) + LK + LMedS geometry", front_end_measure),
                         ("kitti_ba from frames: ORB(10000) + matcher + RANSAC(.99,.05) geometry",
                          lambda c: orb_front_end_measure(c, cpu=(world == 1)))):
            try:                                     # side measurements: a failure here is reported, it does not take the line down
                cfgs[name] = fn(ctx)
            except Exception as e:                   # noqa: BLE001
                cfgs[name] = {"error": "%s: %s" % (type(e).__name__, e)}
        line["configs"] = cfgs

    # ---------------- N > 1: config 3 as written (one sequence sharded, gathered, chained) ---------------
    if world > 1:
        line["strong_scaling"] = strong_scaling_leg(a, ctx, local, world, rank, dist, prm, run)

    if world == 1 and rank == 0 and not a.no_cpu_baseline:
        from oracle import cpu_reference as R
        n = max(8, min(a.cpu_pairs, P))
        cores = os.cpu_count() or 1
        pool = R.CpuPool(seq.kps[:n + 1], seq.descs[:n + 1], seq.K, 8 if a.method == "ransac" else 4, 0.99, a.thr,
                         cores=cores, norm=7 if a.norm == "hamming2" else 6, ratio=None if a.match == "crosscheck" else 0.8)
        pool.run(range(min(n, cores)))
        v, res = pool.run(range(n))
        pool.close()
        # live parity census: cv2's result for these pairs against the GPU's result for the same pairs
        eq = {"n_matches": 0, "n_inliers": 0, "n_good": 0}
        max_rot = 0.0
        for (i, T, nm, ni, ng) in res:
            g = results[i]
            eq["n_matches"] += int(nm == g["n_matches"])
            eq["n_inliers"] += int(ni == g["n_inliers"])
            eq["n_good"] += int(ng == g["n_good"])
            max_rot = max(max_rot, rot_angle(np.asarray(T)[:3, :3], g["T"][:3, :3]))
        line["parity_vs_cv2"] = {"pairs": len(res), "n_matches_equal": eq["n_matches"], "n_inliers_equal": eq["n_inliers"],
                                 "n_good_equal": eq["n_good"], "max_rot_diff_rad": max_rot,
                                 "note": "whole-call comparison on the first pairs of the benchmark sequence; a differing pair "
                                         "is one where cv2's own winning model violates the essential constraints (its "
                                         "unrefined root on an ill-conditioned sample), see tests/test_gpu_cv2_census.py"}
        # SURVEY 8d's other arrangement: one process, OpenCV's own threads over all cores (16 pairs, ~2 s)
        n1 = min(16, n)
        v1 = R.single_process_rate(seq.kps[:n1 + 1], seq.descs[:n1 + 1], seq.K, n1, 8 if a.method == "ransac" else 4, 0.99,
                                   a.thr, threads=cores, norm=7 if a.norm == "hamming2" else 6,
                                   ratio=None if a.match == "crosscheck" else 0.8)
        line["cpu_baseline_single_process"] = {"value": v1, "unit": UNIT, "cores": cores,
                                               "sample": f"first {n1} pairs, one process, cv2.setNumThreads({cores})"}
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores,
                                "kind": "reference" if (R.HAVE_CV2 and R.lm_kind() == "reference") else "port",
                                "sample": f"first {n} pairs of the same sequence; {R.describe()}; {cores} processes x 1 thread",
                                "lm_ms_per_pair": R.lm_ms_per_pair()}
    if rank == 0:
        emit(line)
    run.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
