#!/usr/bin/env python
"""Benchmark of the hot path: correspondence-sets/sec through PointDSC.forward (testing mode).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl engine|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one testing-mode forward over one batch of B synthetic correspondence sets (default: the configuration
BASELINE.json's metric is quoted on, N=1000, B=256 per GPU, 3DMatch snapshot, inlier ratios 0.05/0.1/0.3/0.5 of SURVEY.md §8d).
Batches shard across ranks with no data-path collective (weak scaling: B sets per GPU); NCCL only reduces the timing.

value        : sets/s with inputs resident in HBM (CUDA events around exactly K steps, max over ranks, profiling events OFF)
e2e          : sets/s through the module's streaming loop (model.forward_stream) with pinned HOST tensors — the H2D copy of every
               step's inputs and the D2H copy of its (final_trans, final_labels) are inside the timed region, two calls in flight;
               e2e_sync is the same through K synchronous module calls (nothing overlapped)
roofline     : the dominant kernel (per-layer SC-weighted attention): algorithmic FLOPs per launch / its mean launch duration
               measured live with CUDA events on the launch stream (pdsc_profile_*, a separate profiled pass of K steps)
roofline_stages : every stage of the path against the roofline that bounds it (SURVEY.md §8d formulas)
determinism  : the K timed steps process identical data; their outputs must be bit-identical (asserted)
cpu_baseline : the reference's CPU path on the box's host cores, bounded sample, rank 0 at N=1 only: the UNMODIFIED reference
               module from baseline/_ref when that install is present (kind "reference"), else the torch-CPU restatement in
               oracle/ (kind "port").  `--impl reference` times the same CPU path as its own arm.
extras       : bs=1 latency (the evaluation loops' batch size), BASELINE config D sweep (N in 500..5000, 128 sets per GPU),
               strong scaling of the global B=256 batch when N > 1.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
SNAP_DIRS = {"3dmatch": "PointDSC_3DMatch_release", "kitti": "PointDSC_KITTI_release"}
CTOR = {"3dmatch": dict(inlier_threshold=0.10, sigma_d=0.10, nms_radius=0.10),      # evaluation/test_3DMatch.py:215-224
        "kitti": dict(inlier_threshold=0.6, sigma_d=1.2, nms_radius=0.6)}            # evaluation/test_KITTI.py:166-191
RATIOS = [0.05, 0.1, 0.3, 0.5]     # SURVEY.md §8(d): inlier ratios of the synthetic sets, cycled over the global set index

METRIC = "correspondence-sets/sec (PointDSC.forward, N=1000, B=256)"   # BASELINE.json's metric (the default configuration)
UNIT = "sets/s"


def metric_of(args):
    """BASELINE.json's label at the default configuration, the same label with the actual N and B otherwise (parity-test
    sized runs must not carry the headline label)."""
    return METRIC if (args.n == 1000 and args.batch == 256) else f"correspondence-sets/sec (PointDSC.forward, N={args.n}, B={args.batch})"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--n", type=int, default=1000)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--k", type=int, default=40)
    ap.add_argument("--dataset", default="3dmatch", choices=["3dmatch", "kitti"])
    ap.add_argument("--precision", default=os.environ.get("POINTDSC_PRECISION", "fp16x3"))
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip bs=1 latency / config-D sweep / strong scaling")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (final_trans, final_labels) as DIR/<name>.npy, float32")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "engine":
        ap.error("--dump-outputs writes the engine's outputs: use it with --impl engine")
    return a


def config_of(args, world):
    return {"workload": f"{args.dataset}-like synthetic correspondences, N={args.n}, B={args.batch} sets per GPU per step, "
                        f"k={args.k}, S={int(args.n * 0.1)} seeds, 12 SCNonlocal layers, released {args.dataset} snapshot, "
                        f"inlier ratios {RATIOS} cycled over the global set index",
            "n": args.n, "batch_per_gpu": args.batch, "global_batch": args.batch * world, "k": args.k,
            "precision": args.precision, "parallelism": f"dp{world} (sets sharded, no data-path collective)",
            "l2": "per-step working set exceeds L2 (SC matrix alone is 4*N*NS*B bytes = "
                  f"{4 * args.n * ((args.n + 63) // 64 * 64) * args.batch / 1e6:.0f} MB vs 126 MB L2); no flush needed",
            "profiling": "stage events are OFF in the timed loops of value / e2e; stage shares and rooflines come from a "
                         "separate profiled pass of the same K steps"}


def load_snapshot(dataset):
    import numpy as np
    import torch
    z = np.load(os.path.join(ROOT, "tests", "golden", f"snapshot_{dataset}.npz"))
    return {k: torch.from_numpy(z[k]) for k in z.files}


def make_inputs(n, batch, dataset, rank, world=1):
    """This rank's shard of a global batch of batch*world sets: global set g has seed g and inlier ratio RATIOS[g % 4], so any
    sharding of the same global batch sees the same sets."""
    import torch
    from pointdsc_b200.shard import shard_bounds
    from pointdsc_b200.synth import make_pair
    lo, hi = shard_bounds(batch * world, rank, world)
    pairs = [make_pair(g, n, dataset, RATIOS[g % 4]) for g in range(lo, hi)]
    return {k: torch.stack([p[k] for p in pairs], 0).contiguous() for k in pairs[0]}


class ClockSampler:
    """nvidia-smi clocks/throttle-reason sampler running during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for t, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                mx = float(f[1])
                if t0 <= t <= t1 + 0.1:
                    sm.append(float(f[0]))
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            except ValueError:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------------------------
# the CPU arm: the unmodified reference (baseline/_ref) when installed, else the oracle port
# --------------------------------------------------------------------------------------------------------------------
class CpuPath:
    """One bs=1 testing-mode forward of the reference's CPU implementation per call."""

    def __init__(self, dataset, k=40):
        import torch
        self.torch = torch
        self.kind = None
        ref_model = os.path.join(REF_DIR, "models", "PointDSC.py")
        pkl = os.path.join(REF_DIR, "snapshot", SNAP_DIRS[dataset], "models", "model_best.pkl")
        if os.path.exists(ref_model) and os.path.exists(pkl):
            sys.dont_write_bytecode = True
            if REF_DIR not in sys.path:
                sys.path.insert(0, REF_DIR)
            import models.PointDSC as ref_mod       # the UNMODIFIED reference module (installed copy, see __graft_entry__.install_reference)
            cfg = json.load(open(os.path.join(REF_DIR, "snapshot", SNAP_DIRS[dataset], "config.json")))
            self.model = ref_mod.PointDSC(in_dim=cfg["in_dim"], num_layers=cfg["num_layers"], num_channels=cfg["num_channels"],
                                          num_iterations=cfg["num_iterations"], ratio=cfg["ratio"], k=k, **CTOR[dataset])
            res = self.model.load_state_dict(torch.load(pkl, map_location="cpu"), strict=False)
            assert res.missing_keys == [], res
            self.model.eval()
            self.kind = "reference"
            self.what = "unmodified reference module (baseline/_ref/models/PointDSC.py), released snapshot, eval(), no_grad, fp32"
        else:
            from oracle import pointdsc_oracle as O
            self.O, self.sd = O, load_snapshot(dataset)
            self.cfg = O.default_config(dataset)
            self.cfg["k"] = k
            self.kind = "port"
            self.what = "torch-CPU restatement of the reference (oracle/pointdsc_oracle.py: baseline/_ref is not installed), fp32"

    def forward(self, corr_pos, src, tgt):
        if self.kind == "reference":
            with self.torch.no_grad():
                return self.model({"corr_pos": corr_pos[None], "src_keypts": src[None], "tgt_keypts": tgt[None], "testing": True})
        return self.O.forward_testing(self.sd, self.cfg, corr_pos, src, tgt)


def pick_cpu_threads(cpu, sets):
    """torch's CPU ops on small tensors slow down badly when oversubscribed (128 threads: 26 s per N=1000 forward, 8 threads:
    0.17 s), so "all the host threads it can use" is found by timing three back-to-back forwards per candidate count (bounded: a
    candidate that takes > 4x the best so far ends the search) and keeping the fastest count."""
    import torch
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu})
    best, best_t = cands[0], None
    one = (sets["corr_pos"][0], sets["src_keypts"][0], sets["tgt_keypts"][0])
    for c in cands:
        torch.set_num_threads(c)
        cpu.forward(*one)                     # warm this pool size
        # the SUSTAINED time of three back-to-back forwards (what the measured loop then does), not the fastest single one: one
        # sample, and later the fastest of three, picked 32 threads on boxes where 16 sustain 1.5x more
        t0 = time.perf_counter()
        for _ in range(3):
            cpu.forward(*one)
        dt = (time.perf_counter() - t0) / 3
        if best_t is None or dt < best_t:
            best, best_t = c, dt
        elif dt > 4 * best_t:
            break
    return best


def cpu_rate(cpu, sets, budget_s, threads):
    """sets/s of the CPU path on a bounded sample of the same workload."""
    import torch
    torch.set_num_threads(threads)
    cpu.forward(sets["corr_pos"][0], sets["src_keypts"][0], sets["tgt_keypts"][0])  # warm-up
    done, t0 = 0, time.perf_counter()
    while done < sets["corr_pos"].shape[0] and (time.perf_counter() - t0 < budget_s or done < 2):
        cpu.forward(sets["corr_pos"][done], sets["src_keypts"][done], sets["tgt_keypts"][done])
        done += 1
    dt = time.perf_counter() - t0
    return done / dt, done, dt


def run_reference(args, rank, world):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores, loop of bs=1 testing
    forwards (the reference asserts bs == 1 in testing mode), every step a bounded sample of the workload."""
    if rank != 0:
        return
    import torch
    cpu = CpuPath(args.dataset, args.k)
    probe = make_inputs(args.n, 4, args.dataset, 0)
    threads = pick_cpu_threads(cpu, probe)
    torch.set_num_threads(threads)
    t0 = time.perf_counter()
    cpu.forward(probe["corr_pos"][1], probe["src_keypts"][1], probe["tgt_keypts"][1])
    one = max(time.perf_counter() - t0, 1e-3)
    # a step = a bounded sample of the batch, sized so that steps + warmup stay within ~2 minutes
    per_step = int(max(1, min(args.batch, 120.0 / (one * (args.steps + args.warmup)))))
    need = per_step * (args.steps + args.warmup)
    sets = make_inputs(args.n, min(args.batch, need), args.dataset, 0)
    nsets = sets["corr_pos"].shape[0]

    def step(i):
        for j in range(per_step):
            b = (i * per_step + j) % nsets
            cpu.forward(sets["corr_pos"][b], sets["src_keypts"][b], sets["tgt_keypts"][b])
    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(args.warmup + i)
    dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    sample = (f"{per_step} sets per step (loop of bs=1 testing forwards; the engine's step is {args.batch} sets, rates are per set) "
              f"x {args.steps} steps of the N={args.n} workload, {threads} host threads (fastest of the candidate counts on "
              f"{os.cpu_count()} cores); {cpu.what}")
    cfg = config_of(args, world)
    cfg["reference_sets_per_step"] = per_step
    print(json.dumps({
        "impl": "reference", "metric": metric_of(args), "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": cpu.kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# --------------------------------------------------------------------------------------------------------------------
# per-stage rooflines (SURVEY.md §8d formulas; per rank and per step)
# --------------------------------------------------------------------------------------------------------------------
def stage_rooflines(prof, steps, B, N, k, peaks, sm_count, sm_max_mhz):
    """{stage: {bound, algorithmic work, achieved, peak, frac, ms_per_step}}.  HBM bytes are ALGORITHMIC bytes of the stage as
    designed (what it must read and write once), FLOPs are algorithmic (the fp16x3 format executes 3x the tensor FLOPs)."""
    S, L, C = int(N * 0.1), 12, 128
    KT, QT = (N + 63) // 64, (N + 127) // 128
    hbm = float(peaks.get("hbm_gbs", 6568.4))                 # GB/s, measured copy bandwidth
    tens = float(peaks.get("bf16_tflops_sustained", 1440.5))  # TFLOP/s, measured sustained cuBLAS bf16
    fp32 = sm_count * 128 * 2 * (sm_max_mhz or 1965.0) * 1e6 / 1e12   # TFLOP/s, FFMA lanes x max clock (nominal: no measured fp32 peak)
    T = 10
    rows = {
        "sc": ("hbm", float(B) * KT * QT * 32768, None),                                      # tiled SC write (a1)
        "linear": ("hbm", float(B) * N * (512 + L * 5120), float(B) * N * L * 172032.0),          # layer0 out + per layer: feat in, feat1 out+2 in, Q/K/V images, msg in, feat out
        "attention": ("tensor", float(B) * L * (KT * QT * 32768 + 4.0 * N * 512), float(B) * L * 4.0 * C * N * N),
        "head": ("hbm", float(B) * N * (512 + 512 + 4), float(B) * N * 2.0 * (128 * 32 + 32 * 32 + 32)),
        "seeds": ("fp32", None, float(B) * N * N * 8.0),                                         # N^2 pair tests, ~8 FLOP each
        "knn": ("hbm", float(B) * (N * 512 + 2.0 * S * N * 4), float(B) * 2.0 * S * N * C),      # normed read, S x N distances write + read
        "nsm": ("hbm", float(B) * S * (k * 536 + T * k * 4), float(B) * S * (k * k * C + T * 2.0 * k * k)),   # gather k rows + points, iterates out
        "hypotheses": ("fp32", None, float(B) * S * N * 30.0),
        "refine": ("latency", None, None),
    }
    out = {}
    for name, (bound, nbytes, flops) in rows.items():
        ms = prof[name][0] / steps
        e = {"bound": bound, "ms_per_step": ms, "algorithmic_bytes": nbytes, "algorithmic_flops": flops}
        if ms > 0:
            if nbytes:
                e["achieved_gbs"] = nbytes / (ms * 1e-3) / 1e9
                e["frac_of_hbm_peak"] = e["achieved_gbs"] / hbm
            if flops:
                e["achieved_tflops"] = flops / (ms * 1e-3) / 1e12
                e["frac_of_tensor_peak" if bound in ("tensor", "hbm") else "frac_of_fp32_peak"] = e["achieved_tflops"] / (tens if bound in ("tensor", "hbm") else fp32)
            e["frac"] = {"hbm": e.get("frac_of_hbm_peak"), "tensor": e.get("frac_of_tensor_peak"), "fp32": e.get("frac_of_fp32_peak"),
                         "latency": None}[bound]
        out[name] = e
    out["_peaks"] = {"hbm_gbs": hbm, "tensor_tflops": tens, "fp32_tflops_nominal": fp32,
                     "source": "MEASURED_PEAKS.json (hbm_gbs, bf16_tflops_sustained)" if peaks else "B200_PROFILING.md fallback"}
    return out


def time_steps(model, d, steps, keep=False):
    """CUDA events around exactly `steps` device-resident forwards; returns (ms, outputs of every step if keep)."""
    import torch
    outs = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        o = model.run(d["corr_pos"], d["src_keypts"], d["tgt_keypts"])
        if keep:
            outs.append(o)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), outs


DUMP_BYTES = 64 << 20


def dump_outputs(directory, out, rank, world):
    """`out` (what one step returned) as <directory>/<name>.npy, with a _rank<r> suffix when several ranks write.  Outputs over
    64 MB in all are cut to a seeded sample of the sets, whose indices in the batch are written as sets.npy."""
    import numpy as np
    arrays = {k: v.cpu().numpy() for k, v in out.items()}
    B = len(arrays["final_trans"])
    per_set = sum(a[0].nbytes for a in arrays.values())
    budget = DUMP_BYTES // world - 4096                 # this rank's share, less the .npy headers
    if B * per_set > budget:
        keep = np.sort(np.random.default_rng(0).choice(B, budget // (per_set + 8), replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
        arrays["sets"] = keep.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}{suffix}.npy"), a)


def run_engine(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from pointdsc_b200 import PointDSC
    from pointdsc_b200.shard import gather_counters, output_checksum
    from pointdsc_b200.shard import max_over_ranks as _max_over_ranks
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model = PointDSC(in_dim=6, num_layers=12, num_channels=128, num_iterations=10, ratio=0.1, k=args.k,
                     precision=args.precision, **CTOR[args.dataset])
    res = model.load_state_dict(load_snapshot(args.dataset), strict=False)
    assert res.missing_keys == [], res
    model = model.to(dev).eval()
    B, N = args.batch, args.n
    host = make_inputs(N, B, args.dataset, rank, world)
    pinned = {k: host[k].pin_memory() for k in ("corr_pos", "src_keypts", "tgt_keypts")}
    d = {k: host[k].to(dev) for k in ("corr_pos", "src_keypts", "tgt_keypts")}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        return _max_over_ranks(x, dev)

    # ---- device-resident throughput (profiling events off) -------------------------------------------------------------
    # the clock sampler (an nvidia-smi process) starts BEFORE the warm-up so that its start-up — NVML initialisation takes driver
    # locks for tens of milliseconds — falls into untimed work, and the caching allocator is primed with the K result tensors the
    # timed loop retains for the determinism check (a cudaMalloc inside the timed region stalls the launches behind it: one of
    # three otherwise identical runs lost 36 ms of its 94 ms to such a stall)
    sampler = ClockSampler(local_rank)
    sampler.start()
    prime = [(torch.empty(B, 4, 4, dtype=torch.float32, device=dev), torch.empty(B, N, dtype=torch.float32, device=dev))
             for _ in range(args.steps + 2)]
    del prime
    for _ in range(args.warmup):
        model.run(d["corr_pos"], d["src_keypts"], d["tgt_keypts"])
    # no Python garbage collection inside the timed regions: a generation-2 pass over a process that has imported torch takes tens
    # of milliseconds, i.e. several steps
    import gc
    gc.collect()
    gc.disable()
    barrier()
    t0 = time.perf_counter()
    ms_local, outs = time_steps(model, d, args.steps, keep=True)
    barrier()
    t1 = time.perf_counter()
    gc.enable()
    ms = max_over_ranks(ms_local)
    clocks = sampler.stop(t0, t1)
    value = B * world * args.steps / (ms * 1e-3)
    out = outs[-1]
    # the timed steps process identical data: a race or a read of stale memory would show up as a differing step
    identical = all(torch.equal(o["final_trans"], outs[0]["final_trans"]) and torch.equal(o["final_labels"], outs[0]["final_labels"])
                    for o in outs[1:])
    assert identical, "outputs of the timed steps differ although their inputs are identical"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, rank, world)

    # sanity: the timed work produced registrations (not a skipped / cached forward)
    err = (out["final_trans"].cpu() - host["gt_trans"]).abs().amax(dim=(1, 2))
    scale = 0.05 if args.dataset == "3dmatch" else 0.5
    registered = float((err < scale).float().mean())
    del outs

    # ---- the same K steps with the engine's stage events on: stage shares, per-launch time of the dominant kernel ---------
    model.profile(True)
    time_steps(model, d, args.steps)
    prof = model.profile_read()
    model.profile(False)

    # ---- end to end: pinned host tensors in, host tensors out, every step's copies inside the timed region ---------------
    # (a) the module's streaming loop (model.forward_stream, pdsc_forward_host_submit / _wait): the evaluation drivers' `for data
    #     in loader: model(data)` with two calls in flight, so the H2D copy of step t + 1 and the D2H copy of step t - 1 run beside
    #     the forward of step t.  Every step still copies its own 12 MB in and 1 MB out; the first H2D and the last D2H are exposed.
    # (b) the same K steps as K synchronous module calls (each one H2D -> forward -> D2H -> synchronise): reported as e2e_sync.
    hdata = {"corr_pos": pinned["corr_pos"], "src_keypts": pinned["src_keypts"], "tgt_keypts": pinned["tgt_keypts"], "testing": True}
    for _ in model.forward_stream(hdata for _ in range(min(3, args.warmup))):
        pass
    import numpy as np
    want_t, want_l = out["final_trans"].cpu(), out["final_labels"].cpu()
    want_tn, want_ln = want_t.numpy(), want_l.numpy()
    gc.collect()
    gc.disable()
    barrier()
    th0 = time.perf_counter()
    # every result is read on the host inside the timed region (compared with the device path's) and then dropped, as an
    # evaluation loop does; retaining all K results would time the first touch of K fresh megabytes instead (slow in the
    # GPU boxes' virtual machines: ~4 ms per result)
    streamed, same = 0, True
    for ho in model.forward_stream(hdata for _ in range(args.steps)):
        # numpy, not torch.equal: a torch CPU op fans out over all host cores (128 on the GPU boxes), and waking that thread
        # pool costs milliseconds with a large variance — it cost one run 29 ms of its 93 ms
        same = same and np.array_equal(ho["final_trans"].numpy(), want_tn) and np.array_equal(ho["final_labels"].numpy(), want_ln)
        streamed += 1
    torch.cuda.synchronize()
    th1 = time.perf_counter()
    e2e_s = max_over_ranks(th1 - th0)
    e2e_value = B * world * args.steps / e2e_s
    assert streamed == args.steps and same, "streamed steps differ from the device path"
    h2d = sum(pinned[k].numel() * 4 for k in pinned)
    d2h = ho["final_trans"].numel() * 4 + ho["final_labels"].numel() * 4
    assert torch.equal(ho["final_trans"], out["final_trans"].cpu()) and torch.equal(ho["final_labels"], out["final_labels"].cpu()), \
        "host path and device path disagree"
    for _ in range(min(2, args.warmup)):
        model.run(pinned["corr_pos"], pinned["src_keypts"], pinned["tgt_keypts"])
    barrier()
    ts0 = time.perf_counter()
    for _ in range(args.steps):
        hs = model.run(pinned["corr_pos"], pinned["src_keypts"], pinned["tgt_keypts"])
    torch.cuda.synchronize()
    ts1 = time.perf_counter()
    gc.enable()
    e2e_sync_value = B * world * args.steps / max_over_ranks(ts1 - ts0)
    assert torch.equal(hs["final_trans"], ho["final_trans"]), "synchronous and streamed host paths disagree"

    # ---- extras: bs=1 latency, BASELINE config D sweep, strong scaling -------------------------------------------------
    extras = None
    if not args.no_extras:
        extras = measure_extras(args, model, rank, world, dev, barrier, max_over_ranks)

    counters = output_checksum(out["final_trans"].cpu(), out["final_labels"].cpu())
    counters["registered"] = registered
    per_rank = gather_counters(counters)     # NCCL is used for timing / counters only: there is no data-path collective
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    registered = sum(c["registered"] * c["sets"] for c in per_rank) / max(1.0, sum(c["sets"] for c in per_rank))
    # ---- roofline of the dominant kernel --------------------------------------------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "1400 TFLOP/s sustained (of fallback)"
    attn_ms, attn_launches = prof["attention"]
    flops_per_launch = 4.0 * 128 * N * N * B          # QK^T + PV of one layer over the rank's B sets (algorithmic)
    achieved = flops_per_launch / (attn_ms / max(attn_launches, 1) * 1e-3) / 1e12 if attn_ms > 0 else None
    ns = (N + 63) // 64 * 64
    hbm_bytes = 4.0 * N * ns * B + 4.0 * 128 * N * B * 3 + 4.0 * 128 * N * B   # SC tiles + Q,K,V images (hi+lo) + msg
    hbm_gbs = hbm_bytes / (attn_ms / max(attn_launches, 1) * 1e-3) / 1e9 if attn_ms > 0 else None
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "attention_traffic.json")))
        traffic = tj.get(f"{args.precision}_N{N}_B{B}", {}).get("dram_bytes_per_launch")
    except Exception:
        pass
    executed = {"bf16x3": 3, "fp16x3": 3, "bf16": 1, "fp32": 1}[args.precision]
    roofline = {"kernel": "tc_attention_persistent_kernel" if args.precision != "fp32" else "attention_simt_kernel",
                "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": (achieved / peak_tf) if achieved else None, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_flops_per_launch": flops_per_launch, "launch_ms": attn_ms / max(attn_launches, 1),
                "launches_timed": attn_launches,
                # the same launch seen from the memory side: SC (re-read by every layer) + Q/K/V images + msg
                "hbm_algorithmic_bytes_per_launch": hbm_bytes, "hbm_achieved_gbs": hbm_gbs,
                "hbm_frac_of_copy_peak": (hbm_gbs / float(peaks.get("hbm_gbs", 6568.4))) if hbm_gbs else None,
                "note": f"algorithmic FLOPs = 4*C*N^2*B per layer; {args.precision} executes {executed}x that on the tensor pipe"}
    total_ms = prof["total"][0]
    stages = {k: {"ms_per_step": v[0] / args.steps, "share": (v[0] / total_ms if total_ms > 0 else None)}
              for k, v in prof.items() if k != "total"}
    props = torch.cuda.get_device_properties(dev)
    rstages = stage_rooflines(prof, args.steps, B, N, min(args.k, N - 1), peaks, props.multi_processor_count, clocks.get("sm_max_mhz"))

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpath = CpuPath(args.dataset, args.k)
        threads = pick_cpu_threads(cpath, host)
        rate, done, dt = cpu_rate(cpath, host, args.cpu_seconds, threads)
        cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": cpath.kind,
               "sample": f"first {done} sets of the step's batch, loop of bs=1 testing forwards, {dt:.1f} s on {threads} host threads "
                         f"(fastest of the candidate thread counts on {os.cpu_count()} cores; torch {torch.__version__} CPU); {cpath.what}"}
    launches = model.launches_per_forward(B, N) * args.steps
    e2e_stream = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                  "api": "model.forward_stream(batches): pinned host tensors in, host tensors out, two calls in flight (the copies of "
                         "neighbouring steps overlap the forward; each step's own H2D + D2H are inside the timed region)"}
    e2e_sync = {"value": e2e_sync_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "model(data) per step with pinned host tensors: H2D -> forward -> D2H -> synchronise, nothing overlapped"}
    print(json.dumps({
        "metric": metric_of(args), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"bf16x3": "bf16 hi/lo split (3 products) with f32 accumulate", "bf16": "bf16 with f32 accumulate",
                  "fp16x3": "fp16 hi/lo split (3 products) with f32 accumulate", "fp32": "f32"}[args.precision],
        "data": "synthetic", "config": config_of(args, world),
        # the headline end-to-end number is the faster of the module's two host-tensor entry points, both measured above
        "e2e": dict(e2e_stream if e2e_stream["value"] >= e2e_sync["value"] else e2e_sync),
        "e2e_stream": e2e_stream, "e2e_sync": e2e_sync,
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "roofline_stages": rstages, "cpu_baseline": cpu,
        "stages": stages, "registered_fraction": registered,
        "determinism": {"timed_steps_bit_identical": identical, "steps_compared": args.steps},
        "extras": extras,
        "rank_checksums": [{k: c[k] for k in ("sets", "trans_abs", "inliers")} for c in per_rank]}))
    if world > 1:
        dist.destroy_process_group()


def measure_extras(args, model, rank, world, dev, barrier, max_over_ranks):
    """Bounded extra measurements with the same module (all ranks take part so that barriers match)."""
    import torch
    out = {}
    # (1) bs = 1 latency: the batch size every caller of the reference uses (evaluation/test_3DMatch.py:133, test_KITTI.py:126);
    #     device-resident = pdsc_forward_graph replay, e2e = module call with host tensors (H2D + forward + D2H + sync)
    lat = {}
    for n in (1000, 5000):
        one = make_inputs(n, 1, args.dataset, 0)
        dv = {k: one[k].to(dev) for k in ("corr_pos", "src_keypts", "tgt_keypts")}
        pin = {k: one[k].pin_memory() for k in ("corr_pos", "src_keypts", "tgt_keypts")}
        for _ in range(3):
            model.run(dv["corr_pos"], dv["src_keypts"], dv["tgt_keypts"])
            model.run(pin["corr_pos"], pin["src_keypts"], pin["tgt_keypts"])
        torch.cuda.synchronize()
        reps = 20 if n <= 1000 else 8
        e = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
        e[0].record()
        for i in range(reps):
            model.run(dv["corr_pos"], dv["src_keypts"], dv["tgt_keypts"])
            e[i + 1].record()
        torch.cuda.synchronize()
        dev_ms = statistics.median(e[i].elapsed_time(e[i + 1]) for i in range(reps))
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            model.run(pin["corr_pos"], pin["src_keypts"], pin["tgt_keypts"])
            ts.append((time.perf_counter() - t0) * 1e3)
        # the evaluation loop as the module's streaming loop: host pairs in, host results out, two pairs in flight
        hd = dict(pin, testing=True)
        for _ in model.forward_stream(hd for _ in range(3)):
            pass
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in model.forward_stream(hd for _ in range(4 * reps)):
            pass
        stream_ms = (time.perf_counter() - t0) * 1e3 / (4 * reps)
        lat[f"N{n}"] = {"device_ms_per_pair": dev_ms, "e2e_ms_per_pair": statistics.median(ts), "e2e_stream_ms_per_pair": stream_ms,
                        "reps": reps, "path": "CUDA-graph replay" if n <= model.graph_rows else "eager launches"}
    out["latency_bs1"] = lat
    # (2) BASELINE config D: N in {500, 1000, 2000, 5000}, 1024 sets over 8 GPUs = 128 sets per GPU (weak: per-GPU share)
    sweep = {}
    for n in (500, 1000, 2000, 5000):
        bb = 128
        h = make_inputs(n, bb, args.dataset, rank, world)
        dv = {k: h[k].to(dev) for k in ("corr_pos", "src_keypts", "tgt_keypts")}
        for _ in range(2):
            model.run(dv["corr_pos"], dv["src_keypts"], dv["tgt_keypts"])
        barrier()
        ms, _ = time_steps(model, dv, 5)
        ms = max_over_ranks(ms)
        sweep[f"N{n}"] = {"sets_per_s": bb * world * 5 / (ms * 1e-3), "ms_per_step": ms / 5, "batch_per_gpu": bb, "steps": 5}
        del dv
    out["config_d_sweep"] = sweep
    # (2b) BASELINE.json configs A / B / C as named there (per GPU): A 3DMatch N=1000 B=64; B KITTI N=5000 B=32 (sigma_d 1.2);
    #      C N=2000 with k=80 neighbours, B=256.  B needs the KITTI snapshot: a second module.
    named = {}
    for name, (ds, n, bb, kk) in {"A_3dmatch_N1000_B64": ("3dmatch", 1000, 64, 40), "B_kitti_N5000_B32": ("kitti", 5000, 32, 40),
                                   "C_3dmatch_N2000_k80_B256": ("3dmatch", 2000, 256, 80)}.items():
        if ds == args.dataset:
            mod = model
            mod.k = kk
        else:
            from pointdsc_b200 import PointDSC
            mod = PointDSC(in_dim=6, num_layers=12, num_channels=128, num_iterations=10, ratio=0.1, k=kk, precision=args.precision,
                           **CTOR[ds])
            mod.load_state_dict(load_snapshot(ds), strict=False)
            mod = mod.to(dev).eval()
        h = make_inputs(n, bb, ds, rank, world)
        dv = {k: h[k].to(dev) for k in ("corr_pos", "src_keypts", "tgt_keypts")}
        mod.run(dv["corr_pos"], dv["src_keypts"], dv["tgt_keypts"])
        barrier()
        ms, outs = time_steps(mod, dv, 3, keep=True)
        ms = max_over_ranks(ms)
        err = (outs[-1]["final_trans"].cpu() - h["gt_trans"]).abs().amax(dim=(1, 2))
        named[name] = {"sets_per_s": bb * world * 3 / (ms * 1e-3), "ms_per_step": ms / 3, "batch_per_gpu": bb, "k": kk, "steps": 3,
                       "registered_fraction": float((err < (0.05 if ds == "3dmatch" else 0.5)).float().mean())}
        del dv, outs
        if mod is not model:
            del mod
    model.k = args.k
    out["baseline_configs"] = named
    # (2c) the rows beside the path (SURVEY.md §8f), each timed with CUDA events on rank 0's device (every rank runs them)
    out["next_rows"] = measure_next_rows(model, dev)
    # (3) strong scaling: the global B = 256 batch split over the ranks
    if world > 1:
        bb = max(1, 256 // world)
        h = make_inputs(args.n, bb, args.dataset, rank, world)
        dv = {k: h[k].to(dev) for k in ("corr_pos", "src_keypts", "tgt_keypts")}
        for _ in range(2):
            model.run(dv["corr_pos"], dv["src_keypts"], dv["tgt_keypts"])
        barrier()
        ms, _ = time_steps(model, dv, 10)
        ms = max_over_ranks(ms)
        out["strong_scaling"] = {"global_batch": bb * world, "batch_per_gpu": bb, "sets_per_s": bb * world * 10 / (ms * 1e-3),
                                 "ms_per_step": ms / 10, "steps": 10}
    return out


def measure_next_rows(model, dev):
    """f1 (front end), f2 (descriptors), f3 (evaluation statistics), f4 (non-testing forward with M, N x N power iteration): milliseconds per call
    and the achieved rate against the bound that applies (algorithmic bytes or FLOPs)."""
    import torch
    from pointdsc_b200.frontend import match
    from pointdsc_b200.metrics import eval_stats
    from pointdsc_b200.spectral import leading_eigenvector
    from pointdsc_b200.synth import make_batch

    def timed(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps
    res = {}
    g = torch.Generator().manual_seed(0)
    ns = nt = 5000
    sd = torch.nn.functional.normalize(torch.randn(ns, 32, generator=g), dim=1).to(dev)
    td = torch.nn.functional.normalize(torch.randn(nt, 32, generator=g), dim=1).to(dev)
    sk, tk = torch.rand(ns, 3, generator=g).to(dev), torch.rand(nt, 3, generator=g).to(dev)
    for mutual in (False, True):
        ms = timed(lambda: match(sd, td, sk, tk, use_mutual=mutual))
        flops = 2.0 * ns * nt * 32 * (2 if mutual else 1)
        res[f"f1_match_fcgf32_Ns5000_Nt5000_mutual{int(mutual)}"] = {"ms": ms, "bound": "fp32", "achieved_tflops": flops / (ms * 1e-3) / 1e12,
                                                                     "note": "includes the 4-byte device->host read of the correspondence count"}
    b = make_batch(range(8), 1000, "3dmatch", 0.3)
    B = 256
    rep = {k: b[k].repeat(B // 8, *([1] * (b[k].dim() - 1))).to(dev) for k in ("src_keypts", "tgt_keypts", "gt_trans", "gt_labels")}
    lab = (torch.rand(B, 1000, generator=g) < 0.3).float().to(dev)
    ms = timed(lambda: eval_stats(rep["gt_trans"], rep["gt_trans"], rep["src_keypts"], rep["tgt_keypts"], lab, rep["gt_labels"]))
    res["f3_eval_stats_B256_N1000"] = {"ms": ms, "bound": "hbm", "achieved_gbs": B * 1000 * 32.0 / (ms * 1e-3) / 1e9,
                                       "note": "8 MB of inputs: launch-latency bound"}
    n = 5000
    pts = torch.rand(n, 3, generator=g) * 3
    ds = torch.cdist(pts, pts)
    m = torch.clamp(1 - (ds - ds.t().roll(1, 0)) ** 2, min=0)[None].contiguous().to(dev)
    ms = timed(lambda: leading_eigenvector(m, num_iterations=10, early_exit=False), reps=3)
    res["f4_leading_eigenvector_N5000_10iters"] = {"ms": ms, "bound": "hbm (L2-resident: 100 MB matrix re-read by every iteration)",
                                                   "achieved_gbs": 10 * 4.0 * n * n / (ms * 1e-3) / 1e9}
    bb = make_batch(range(16), 1000, "3dmatch", 0.3)
    dv = [bb[k].to(dev) for k in ("corr_pos", "src_keypts", "tgt_keypts")]
    was = model.training
    model.eval()
    ms = timed(lambda: model.run_eval(*dv, want_M=True), reps=3)
    res["f4_forward_without_testing_key_B16_N1000_with_M"] = {"ms": ms, "sets_per_s": 16 / (ms * 1e-3)}
    model.train(was)
    # f2: a 3DMatch-fragment-sized synthetic scene (300 k points -> ~5 k key points at 5 cm), stage by stage
    from pointdsc_b200 import descriptors as D
    from pointdsc_b200.synth_scene import scene
    cloud = torch.from_numpy(scene(300000, seed=0)).to(dev)
    voxel = 0.05
    kp = D.voxel_down_sample(cloud, voxel)
    nrm = D.estimate_normals(kp, 2 * voxel, 30)
    m = int(kp.shape[0])
    res["f2_voxel_down_sample_n300k_5cm"] = {"ms": timed(lambda: D.voxel_down_sample(cloud, voxel)), "key_points": m,
                                              "note": "includes the device->host read of the key-point count"}
    res["f2_estimate_normals"] = {"ms": timed(lambda: D.estimate_normals(kp, 2 * voxel, 30)), "points": m, "distance_evaluations": m * m}
    res["f2_compute_fpfh"] = {"ms": timed(lambda: D.compute_fpfh(kp, nrm, 5 * voxel, 100, normalise=True)), "points": m,
                              "distance_evaluations": m * m}
    return res


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import __graft_entry__ as g
    g.build()   # no-op unless the sources changed since the in-tree library was built
    run_engine(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
