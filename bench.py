"""bench.py -- SAC grad-steps/sec (batch 256, 64x64 depth) on N B200s.

  python bench.py --gpus N --steps K --warmup W             (N>1: launched under torchrun)
  python bench.py --impl reference ...                      (CPU arm: the oracle restatement of
                                                             SB2.10.1/TF1.14's SAC step, all host cores)

A "step" = one SAC minibatch gradient step (replay sample -> VecNormalize -> 3 CNN fwd, 2 CNN bwd,
heads, losses -> [all-reduce] -> 3x Adam -> Polyak) at batch 256 per GPU on synthetic 64x64x2 depth
observations (BASELINE.json configs[1]).  `value` times K steps with the replay already resident in
HBM (CUDA events, max over ranks); `e2e` times the same step through the C-ABI parity entry point
with HOST (pinned) batches, i.e. host->device copies of the batch and device->host read of the
losses inside the timed region.  Weak scaling: every rank processes its own 256-sample minibatch
and one NCCL all-reduce averages the gradients, so N ranks = one step on a global batch of N*256;
value = N x synchronous steps/s, in 256-sample step equivalents (SURVEY.md section 8e).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# The driver reads ONE JSON line on stdout.  NCCL (and anything else native) prints its banners to fd 1, so fd 1 is pointed at stderr
# for the whole run and the JSON line goes to the saved descriptor.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: str):
    os.write(_REAL_STDOUT, (line.rstrip("\n") + "\n").encode())
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")
FLOP_PER_STEP_B256 = 2 * 256 * 18_923_328          # SURVEY.md section 8d: 9.689 GFLOP
LR = 3e-4
KERNEL_DESC = ("cg_kernel (TMA-fed tcgen05 contraction engine, csrc/cg.cu): converged producer warps issue cp.async.bulk.tensor boxes -- "
               "implicit-im2col / shifted-window / zero-bordered tensor-map views of the BF16 activation planes, all planes of an operand in one "
               "box -- into a 128B-swizzled smem ring; tcgen05.mma kind::f16 with fp32 TMEM accumulators, one wide MMA per operand plane; "
               "forward = 6-product 3-plane split, backward = 3-product 2-plane split; TWO persistent launches per step (forward chain "
               "conv1..fc0, backward chain heads dgrad..conv wgrads), layers chained tile by tile through arrival counters")
WORKLOAD = "SAC depth CNN (config/gripper_grasp.yaml), batch 256/GPU, 64x64x2 obs, 1M-slot replay"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["bf16_tflops"], d["hbm_gbs"], "measured (MEASURED_PEAKS.json, burst)"
    return 1590.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons streamed (-lms 100) DURING the timed region."""

    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.dev, self.rows, self.proc = dev, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.dev), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
                out = ""
            self.rows = [[x.strip() for x in line.split(",")] for line in out.splitlines() if line.count(",") >= 5]

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def load_case():
    from oracle import sac_ref as R  # only used by the cpu_baseline / reference legs
    vn = dict(np.load(os.path.join(GOLD, "vecnorm_sac_depth.npz")))
    raw = dict(np.load(os.path.join(GOLD, "sac_depth_params.npz")))
    cfg = R.SACConfig(obs_shape=(64, 64, 2))
    params = {n: raw[n] for n, _ in R.param_specs(cfg)}
    return cfg, params, vn


def cpu_reference_steps(batch, seconds=None, threads=None, steps=None, warmup=1):
    """Times the CPU restatement of the SB2 SAC step (oracle/sac_ref.py, PyTorch-CPU fp32).

    The thread count is calibrated first (one timed step per candidate): on many-core hosts the
    small per-layer ops of this graph run far slower with every hardware thread than with a
    moderate pool, and TF1's own intra-op pool would be tuned the same way.  Either a time budget
    (`seconds`, capped at 400 steps) or an exact step count (`steps`) bounds the sample.
    Returns (steps/s, steps, seconds, threads_used)."""
    import torch
    from oracle import sac_ref as R
    from b200grasp import synth
    cfg, params, vn = load_case()
    raw = synth.make_transitions(batch, vn["obs_mean"], vn["obs_var"])
    norm = dict(obs=R.normalize_obs(raw["obs"], vn["obs_mean"], vn["obs_var"]),
                next_obs=R.normalize_obs(raw["next_obs"], vn["obs_mean"], vn["obs_var"]),
                act=raw["act"], rew=R.normalize_reward(raw["rew"], float(vn["ret_var"])), done=raw["done"])
    eps = synth.make_eps(batch)
    p, opt = params, R.OptState.zeros(params)
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    if threads is None:
        cands = sorted({c for c in (avail, 64, 32, 16, 8) if c <= avail}, reverse=True)
        best, best_t = cands[-1], float("inf")
        for c in reversed(cands):                  # small pools first: they bound the calibration time
            torch.set_num_threads(c)
            R.sac_step(p, opt, norm, eps, LR, cfg, torch.float32)
            t0 = time.perf_counter()
            R.sac_step(p, opt, norm, eps, LR, cfg, torch.float32)
            dt = time.perf_counter() - t0
            if dt < best_t:
                best, best_t = c, dt
            if dt > 4 * best_t:
                break
        threads = best
    torch.set_num_threads(threads)
    for _ in range(max(1, warmup)):
        _, _, p, opt = R.sac_step(p, opt, norm, eps, LR, cfg, torch.float32)
    n, t0 = 0, time.perf_counter()
    while True:
        _, _, p, opt = R.sac_step(p, opt, norm, eps, LR, cfg, torch.float32)
        n += 1
        el = time.perf_counter() - t0
        if steps is not None:
            if n >= steps:
                break
        elif el >= seconds or n >= 400:
            break
    return n / el, n, el, threads


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path cannot run here
    (stable-baselines 2.10.1 / TF 1.14 are not installable, SURVEY.md section 8c), so this arm times
    the oracle port on the host cores: W warm-up steps, then EXACTLY K timed B=256 steps.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rate, n, el, cores = cpu_reference_steps(256, steps=max(1, args.steps), warmup=max(1, min(args.warmup, 5)))
    line = {
        "impl": "reference", "metric": "SAC grad-steps/sec (batch 256, 64x64 depth)", "value": rate, "unit": "steps/s",
        "n_gpus": args.gpus, "steps": n, "warmup": max(1, min(args.warmup, 5)), "ms_per_step": 1e3 / rate, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": 256, "parallelism": "cpu",
                   "note": "CPU restatement of SB2.10.1/TF1.14 SAC step (oracle/sac_ref.py, PyTorch-CPU fp32), not TF itself; "
                           "one fixed pre-normalised B=256 batch (no replay sampling / VecNormalize inside the step: favours the CPU arm)"},
        "cpu_baseline": {"value": rate, "unit": "steps/s", "cores": cores, "kind": "port",
                         "sample": f"{n} full B=256 gradient steps in {el:.1f}s; torch intra-op threads calibrated to {cores} of {os.cpu_count()}"},
        "e2e": {"value": rate, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(json.dumps(line))


def numa_bind(dev):
    """Binds this process to the host CPUs local to GPU `dev` (sysfs local_cpulist of its PCI function) BEFORE the
    pinned e2e buffers are allocated, so that their pages and the copy-issuing thread sit on the GPU's NUMA node.
    Best effort: returns a description for the JSON line."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=20).stdout.strip().lower()
        bus = out[-12:] if len(out) >= 12 else out           # 00000000:1b:00.0 -> 0000:1b:00.0
        path = f"/sys/bus/pci/devices/{bus}/local_cpulist"
        cpus = set()
        for part in open(path).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            node = open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip()
            return f"bound to {len(cpus)} cpus local to {bus} (numa node {node})"
    except Exception as e:                                   # noqa: BLE001
        return f"not bound ({type(e).__name__})"
    return "not bound (no local cpu list)"


def fill_replay(L, vn, n_fill, rank, distinct_chunks=8, chunk=2048):
    """`n_fill` transitions into the device replay: `distinct_chunks` x `chunk` seeded synthetic transitions generated
    on the host, cycled until n_fill slots are written (values only matter for the parity legs; the working set, the
    DRAM page spread and the random per-step slot draw are what the timing sees)."""
    from b200grasp import synth
    cache, i = [], 0
    while i < n_fill:
        k = (i // chunk) % distinct_chunks
        if k >= len(cache):
            cache.append(synth.make_transitions(chunk, vn["obs_mean"], vn["obs_var"], seed=synth.DATA_SEED + 1000 * rank + k))
        tr = cache[k]
        n = min(chunk, n_fill - i)
        L.replay_add(tr["obs"][:n], tr["act"][:n], tr["rew"][:n], tr["next_obs"][:n], tr["done"][:n])
        i += n


def dump_outputs(out_dir, metrics, batch, params):
    """Writes what the last timed step hands a caller, one .npy per array: its losses and statistics (float64 scalars,
    named as b2g_sac_metrics), the per-sample outputs of its minibatch together with the replay slots and policy noise it
    drew (batch_*, so that identical inputs can be confirmed), and the parameters it left (param_*, '/' written as '__').
    The step reduces with float atomics, so two runs on identical inputs are not bit-identical: on a B200 (1000 W limit) they
    agreed to 4e-6 relative after 23 updates, while after 220 updates Adam had grown the differences to the size of the values.
    Compare builds at a small --warmup + --steps."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.float64(v) for k, v in metrics.items()}
    arrays.update({"batch_" + k: np.asarray(v, np.float64 if k == "indices" else np.float32) for k, v in batch.items()})
    arrays.update({"param_" + n.replace("/", "__"): np.asarray(a, np.float32) for n, a in params.items()})
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--replay-filled", type=int, default=65536, help="transitions resident in HBM (2 x 32 KiB each: 4 GiB >> 126 MB L2)")
    ap.add_argument("--buffer-size", type=int, default=1_000_000)
    ap.add_argument("--regions", type=int, default=7, help="the K timed steps are split into this many regions; the MEDIAN region is reported")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dp", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1: p2p = the optimiser launch reduces / updates / broadcasts over NVLink peer memory; nccl = all-reduce + replicated Adam")
    ap.add_argument("--no-c3", action="store_true", help="skip the RGB-D B=1024 extra measurement (config.extra.c3)")
    ap.add_argument("--precision", default="bf16x3", choices=["fp32", "bf16x3", "bf16"],
                    help="bf16x3 = tcgen05 BF16 hi/lo split, the mode that passes the 1e-4 parity tests (default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's losses, per-sample outputs and updated parameters to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    args.regions = max(args.regions, 5)

    import torch
    import torch.distributed as dist
    import b200grasp
    from b200grasp import synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = numa_bind(local)                      # before any pinned allocation / CUDA context thread
    torch.cuda.set_device(local)
    nccl_id = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(b200grasp.Learner.nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        nccl_id = bytes(idt.cpu().numpy().tobytes())

    vn = dict(np.load(os.path.join(GOLD, "vecnorm_sac_depth.npz")))
    raw_params = dict(np.load(os.path.join(GOLD, "sac_depth_params.npz")))
    B = args.batch
    prec = {"fp32": 0, "bf16x3": 1, "bf16": 2}[args.precision]
    L = b200grasp.Learner((64, 64, 2), n_act=5, batch_size=B, buffer_size=args.buffer_size, seed=1234, device=local,
                          rank=rank, nranks=world, nccl_id=nccl_id, precision=prec)
    if world > 1 and args.dp == "p2p":
        L.dp_connect_torch()
    L.load_parameters(raw_params)      # identical replicas on every rank
    L.set_norm_stats(vn["obs_mean"], vn["obs_var"], float(vn["ret_var"]), float(vn["clip_obs"]), float(vn["clip_reward"]),
                     float(vn["epsilon"]))
    # replay shard of this rank (different data per rank), resident in HBM before the timed region
    fill_replay(L, vn, args.replay_filled, rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(vals):
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.cpu()]

    # ---- parity_n (outside every timed region): first-step losses of the N-rank learner on a seeded N*B batch (each rank
    # takes its slice through the C ABI, gradients and losses are averaged by the step's own collective) against the
    # ORACLE's single step on the concatenated batch (SURVEY.md section 8e); replica identity is checked after the run.
    parity = None
    if prec != 2:
        trp = synth.make_transitions(B * world, vn["obs_mean"], vn["obs_var"], seed=4242)
        epsp = synth.make_eps(B * world, seed=4243)
        sl = slice(rank * B, (rank + 1) * B)
        outp = L.step_explicit(trp["obs"][sl], trp["act"][sl], trp["rew"][sl], trp["next_obs"][sl], trp["done"][sl], epsp[sl], lr=LR,
                               apply_update=False)
        if rank == 0:
            from oracle import sac_ref as R          # the checker, never the thing measured
            cfgp = R.SACConfig(obs_shape=(64, 64, 2))
            pp = {n: raw_params[n] for n, _ in R.param_specs(cfgp)}
            normp = dict(obs=R.normalize_obs(trp["obs"], vn["obs_mean"], vn["obs_var"]),
                         next_obs=R.normalize_obs(trp["next_obs"], vn["obs_mean"], vn["obs_var"]), act=trp["act"],
                         rew=R.normalize_reward(trp["rew"], float(vn["ret_var"])), done=trp["done"])
            refp, _, _, _ = R.sac_step(pp, R.OptState.zeros(pp), normp, epsp, LR, cfgp, torch.float64)
            keys = ("policy_loss", "qf1_loss", "qf2_loss", "value_loss", "grad_norm_pi", "grad_norm_values")
            errs = {k: abs(outp[k] - float(refp[k])) / abs(float(refp[k])) for k in keys}
            q_err = float(np.linalg.norm(outp["q1"] - np.asarray(refp["q1"]).reshape(-1)[sl]) / np.linalg.norm(np.asarray(refp["q1"]).reshape(-1)[sl]))
            parity = {"oracle_batch": B * world, "rel_err": {k: float(f"{v:.3g}") for k, v in errs.items()}, "q1_rel_err_rank0": float(f"{q_err:.3g}"),
                      "tol": 1e-4, "first_step_ok": bool(max(errs.values()) <= 1e-4 and q_err <= 1e-4)}

    # ---- device-resident throughput: exactly K graph replays, split into R regions of near-equal size, CUDA events on the
    # learner's stream (b2g_sac_step brackets a region's launches with events), barrier + synchronize on both sides of every
    # region, max over ranks per region, MEDIAN per-step time over regions.  Inputs: random slots of a replay working set far
    # larger than L2.
    n_regions = min(args.regions, args.steps)
    sizes = [args.steps // n_regions + (i < args.steps % n_regions) for i in range(n_regions)]
    L.step(args.warmup, lr=LR)
    barrier()
    region_ms = []
    with ClockSampler(local) as clk:
        time.sleep(0.25)                       # let the sampler stream before the timed regions start
        for n in sizes:
            barrier()
            last = L.step(n, lr=LR)            # one timed region
            region_ms.append(L.last_step_ms())
        barrier()
    region_ms = max_over_ranks(region_ms)
    ms_step = float(np.median([t / n for t, n in zip(region_ms, sizes)]))
    sync_steps_per_s = 1e3 / ms_step
    value = world * sync_steps_per_s
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, L.last_batch(), L.get_parameters())

    # ---- end to end through the C ABI with pinned HOST batches (H2D of the batch + D2H of the losses per step)
    tr = synth.make_transitions(B, vn["obs_mean"], vn["obs_var"], seed=77 + rank)
    eps = synth.make_eps(B, seed=78 + rank)
    pin = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory().numpy() for k, v in dict(tr, eps=eps).items()}
    host_batch = sum(v.nbytes for v in pin.values())          # what the caller hands over (full observations)
    # what crosses PCIe: the library compacts each observation on the host (image planes + the one actuator value: the constant
    # actuator plane is never read beyond pixel [0,0]) into pinned staging and copies that
    h2d = 2 * B * (64 * 64 * 1 + 4) * 4 + sum(pin[k].nbytes for k in ("act", "rew", "done", "eps"))
    e2e_steps = max(10, min(args.steps, 200))
    for _ in range(3):
        L.step_host_pipelined(pin["obs"], pin["act"], pin["rew"], pin["next_obs"], pin["done"], pin["eps"], lr=LR)
    L.pipeline_flush()
    e2e_runs = []
    for _ in range(3):
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):    # every step: H2D of its batch (pinned) + D2H of a step's losses; copy k overlaps compute k-1
            L.step_host_pipelined(pin["obs"], pin["act"], pin["rew"], pin["next_obs"], pin["done"], pin["eps"], lr=LR)
        last = L.pipeline_flush()
        torch.cuda.synchronize()
        e2e_runs.append(time.perf_counter() - t0)
        assert np.isfinite(last["qf1_loss"])
    el = float(np.median(max_over_ranks(e2e_runs)))
    e2e = world * e2e_steps / el
    # raw host->device rate of the same pinned buffers (what bounds e2e on a PCIe box)
    dbuf = torch.empty(pin["obs"].nbytes // 4, dtype=torch.float32, device="cuda")
    src = torch.from_numpy(pin["obs"]).reshape(-1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(20):
        dbuf.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    h2d_gbs = 20 * pin["obs"].nbytes / (time.perf_counter() - t0) / 1e9
    # un-pipelined variant of the same call (b2g_sac_step_explicit: copy, step, read back, return)
    t0 = time.perf_counter()
    for _ in range(max(10, e2e_steps // 4)):
        L.step_explicit(pin["obs"], pin["act"], pin["rew"], pin["next_obs"], pin["done"], pin["eps"], lr=LR)
    e2e_sync = world * max(10, e2e_steps // 4) / (time.perf_counter() - t0)
    # the learn() loop of the SB-shaped front end: one new transition enters the device replay per gradient step
    one = {k: v[:1] for k, v in pin.items() if k != "eps"}
    t0 = time.perf_counter()
    for it in range(e2e_steps):
        L.replay_add(one["obs"], one["act"], one["rew"], one["next_obs"], one["done"])
        L.step_async(1, lr=LR)                    # what SAC.learn does: enqueue, read the losses back when they are logged
        if it % 100 == 99:
            L.step(0, lr=LR)
    L.step(0, lr=LR)
    e2e_learn = world * e2e_steps / (time.perf_counter() - t0)

    # ---- replica identity after everything above (hundreds of updates): byte-identical parameters on every rank
    if parity is not None or world > 1:
        import hashlib
        dig = hashlib.sha1(b"".join(a.tobytes() for a in L.get_parameters().values())).hexdigest()
        digs = [dig]
        if world > 1:
            digs = [None] * world
            dist.all_gather_object(digs, dig)
        if rank == 0 and parity is not None:
            parity["replicas_identical"] = bool(all(d == digs[0] for d in digs))
            parity["ranks"] = world

    # ---- dominant-kernel roofline: per-launch device time of every group of ONE step (CUDA events on
    # the learner's stream between launches, serial issue), on rank 0.  The tensor-engine launches' SHARE of that serial
    # profile is applied to the graph-mode ms_per_step, so launch_ms can never exceed the timed step.
    line = None
    prof = None
    for _ in range(3):              # every rank: the step contains the all-reduce
        prof = L.profile_step(lr=LR)
    launches_per_step = L.launches_per_step()
    L.close()

    c3 = None
    if rank == 0 and world == 1 and not args.no_c3 and prec != 0:
        # BASELINE.json configs[2]: SAC RGB-D (64x64x4 image + feature plane), batch 1024, one B200
        vn5 = dict(np.load(os.path.join(GOLD, "vecnorm_sac_rgbd.npz")))
        L3 = b200grasp.Learner((64, 64, 5), n_act=5, batch_size=1024, buffer_size=8192, seed=99, device=local, precision=prec)
        L3.set_norm_stats(vn5["obs_mean"], vn5["obs_var"], float(vn5["ret_var"]), float(vn5["clip_obs"]), float(vn5["clip_reward"]),
                          float(vn5["epsilon"]))
        for i in range(4):
            t5 = synth.make_transitions(2048, vn5["obs_mean"], vn5["obs_var"], seed=31 + i)
            L3.replay_add(t5["obs"], t5["act"], t5["rew"], t5["next_obs"], t5["done"])
        k3 = max(20, args.steps // 4)
        L3.step(max(3, args.warmup // 2), lr=LR)
        r3 = []
        for _ in range(5):
            torch.cuda.synchronize()
            L3.step(k3, lr=LR)
            r3.append(L3.last_step_ms())
        ms3 = float(np.median(r3)) / k3
        flops3 = 2 * 1024 * 25_835_328
        peak_tf, _, _ = peaks()
        c3 = {"workload": "SAC RGB-D CNN (config/full_depth_obs.yaml shapes), batch 1024, 64x64x5 obs, 8192 resident transitions (1.3 GiB)",
              "value": 1e3 / ms3, "unit": "steps/s (batch-1024 steps)", "ms_per_step": ms3, "steps": k3, "regions": 5,
              "flop_per_step": flops3, "tensor_frac_whole_step": flops3 / (ms3 * 1e-3) / 1e12 / peak_tf}
        L3.close()

    if rank == 0:
        gemm_groups = {k: v for k, v in prof.items() if "fused" in k or k.startswith("conv") or k.startswith("cnn_") or k.startswith("fc1_")
                       or k.startswith("heads_fc0") or k == "heads_dgrad" or (k == "heads_wgrad" and "fwd_fused" not in prof)}
        gemm_serial = sum(gemm_groups.values())
        share = gemm_serial / sum(prof.values())
        gemm_ms = share * ms_step
        peak_tf, peak_hbm, peak_src = peaks()
        flops = FLOP_PER_STEP_B256 * B / 256
        achieved = flops / (gemm_ms * 1e-3) / 1e12
        traffic = None
        tnote = None
        for tname in ("traffic_r2.json", "traffic_r1.json"):
            tpath = os.path.join(ROOT, "profiles", tname)
            if os.path.exists(tpath):          # dram read+write per tensor-engine launch from the committed ncu --set full capture
                tj = json.load(open(tpath))
                traffic = tj.get("dram_bytes_per_launch", tj.get("gg_tc_kernel_dram_bytes_per_launch"))
                tnote = f"profiles/{tname}: ncu dram__bytes_read.sum + dram__bytes_write.sum per tensor-engine launch (mean over the step's launches)"
                break
        roofline = {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                    "traffic": traffic, "traffic_unit": tnote,
                    "kernel": KERNEL_DESC if prec else "gg_simt_kernel (fp32 FFMA engine)",
                    "peak_source": peak_src, "launch_ms": gemm_ms, "launches": len(gemm_groups),
                    "launch_ms_note": "tensor-engine share of the serial per-launch profile x graph-mode ms_per_step",
                    "step_share": share, "per_group_ms_serial": {k: round(v, 4) for k, v in prof.items()},
                    "whole_step_frac": value / world * flops / 1e12 / peak_tf,
                    "hbm_algorithmic_gbs": 62.0e6 / (ms_step * 1e-3) / 1e9, "hbm_frac_of_measured": 62.0e6 / (ms_step * 1e-3) / 1e9 / peak_hbm}
        cpu = None
        if not args.no_cpu_baseline:
            rate, n, cel, cores = cpu_reference_steps(B, args.cpu_seconds)
            cpu = {"value": rate, "unit": "steps/s", "cores": cores, "kind": "port",
                   "sample": f"{n} full B={B} gradient steps in {cel:.1f}s (oracle/sac_ref.py, PyTorch-CPU fp32)"}
        line = {
            "metric": "SAC grad-steps/sec (batch 256, 64x64 depth)", "value": value, "unit": "steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "f32", "bf16x3": "bf16x3 (fp32-faithful split, f32 accumulate)", "bf16": "bf16"}[args.precision], "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "global_batch": B * world, "replay_capacity": args.buffer_size, "replay_filled": args.replay_filled,
                       "l2": f"inputs larger than L2: replay working set {args.replay_filled * 2 * 32768 / 2**30:.1f} GiB >> 126 MB; minibatch slots are random per step",
                       "timing": f"{args.steps} steps in {n_regions} regions of {sizes} steps, median per-step time over regions (CUDA events on the learner's stream, max over ranks per region); regions_ms={[round(x, 3) for x in region_ms]}",
                       "precision": {"fp32": "fp32 FFMA (B2G_PREC_FP32_SIMT)", "bf16x3": "tcgen05 BF16 hi/lo split x3, fp32 TMEM accumulate (B2G_PREC_BF16X3; passes 1e-4 parity)", "bf16": "tcgen05 single-pass BF16 (fast mode, ~5e-4 on Q)"}[args.precision], "parallelism": f"dp{world}" + ("" if world == 1 else (" (gradients reduced, slices updated and parameters broadcast by one kernel over NVLink peer memory)" if args.dp == "p2p" else " (NCCL all-reduce, replicated Adam)")),
                       "sync_steps_per_s": sync_steps_per_s, "numa": numa,
                       "extra": {"c3": c3}},
            "clocks": clk.summary(),
            "e2e": {"value": e2e, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 16 * 4 + 8 + 64, "steps": e2e_steps,
                    "host_batch_bytes_per_step": host_batch, "api": "b2g_sac_step_host_pipelined: full 256-sample HOST batch every step (compacted by the library on 16 host threads, copied from its pinned staging), losses read back every step (one step late); median of 3 runs",
                    "h2d_gbs_achieved": h2d_gbs, "h2d_bound_steps_per_s": h2d_gbs * 1e9 / h2d,
                    "unpipelined_steps_per_s": e2e_sync,
                    "learn_loop_steps_per_s": e2e_learn, "learn_loop_h2d_bytes_per_step": int(sum(v.nbytes for v in one.values()))},
            "gpu_launches": launches_per_step * args.steps,
            "parity_n": parity,
            "roofline": roofline, "cpu_baseline": cpu,
        }
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        emit(json.dumps(line))


if __name__ == "__main__":
    main()
