#!/usr/bin/env python
"""bench.py -- MLPG frames/s on BASELINE.json configs[1] (batched MLPG, 256 utterances T~600,
D=187 Merlin layout, 3 windows, per-frame diagonal variances, float32 in / float64 arithmetic).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One step = one pass of the hot path (banded W^T S^-1 W assemble + factor + solve for every static
dimension of every utterance) over one batch of synthetic input.  Prints ONE JSON line (rank 0).

  value     : whole-job frames/s with the inputs already resident in HBM (CUDA events, max over ranks)
  e2e       : the same metric through the public host-buffer API (nnmnkwii_b200.paramgen.mlpg_batch
              on pinned NumPy arrays -> C ABI nnk_mlpg_batch_host): H2D + solve + D2H every step
  roofline  : algorithmic bytes of the dominant kernel / its CUDA-event duration vs MEASURED_PEAKS.json
  cpu_baseline : the reference's own CPU path (oracle/_ref = unmodified nnmnkwii, per utterance and per
              stream paramgen.mlpg as in its gallery notebooks) on this box's host cores
  --impl reference : times that CPU path only (rank 0), same metric/config/unit.

Multi-GPU (torchrun, one rank per GPU, --gpus N > 1): BASELINE.json configs[4] -- the 8192-utterance
ragged batch (T ~ U{200..2000}, 9.0e6 frames, D=187) STRONG-scaled over the ranks through
nnmnkwii_b200.sharding (ShardPlan -> pre-sharded device buffers -> per bucket: solve, then in-place NCCL
all-gather on a side stream while the next bucket solves).  One step = one full pass: every solve AND
every all-gather, every step (nothing is amortised over --steps).  The line reports kernel ms, exposed
all-gather ms and their sum.  The N=1 line carries `scale_workload`: the same 8192-utterance pass on
one GPU, the denominator for the scaling efficiency of the N>1 lines.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_UTT = 256
T_LO, T_HI = 540, 660
D_IN, D_OUT = 187, 63
ALGO_BYTES_PER_FRAME = 1744  # SURVEY.md 8(d): 186 cols mean + 186 cols variance in, 62 out, vuv copy 4+4 (f32)
WINDOWS = [(0, 0, np.array([1.0])), (1, 1, np.array([-0.5, 0.0, 0.5])), (1, 1, np.array([1.0, -2.0, 1.0]))]
# ncu --set full summaries of the dominant kernel on configs[1] (newest round first): roofline.traffic is parsed from them
DOMINANT_PROFILES = ["r02_mlpg_dominant_cfg2*_ncu.txt", "r01_mlpg_v11_as_3a_l2pf_ncu.txt"]
METRIC = "mlpg_frames_per_sec"
UNIT = "frames/s"


def make_batch(rank):
    rng = np.random.default_rng(1234 + rank)
    lens = rng.integers(T_LO, T_HI + 1, size=N_UTT)
    n = int(lens.sum())
    means = rng.random((n, D_IN), dtype=np.float32)
    variances = rng.random((n, D_IN), dtype=np.float32) + np.float32(0.1)
    return lens, means, variances


def config(n_gpus):
    return {
        "workload": "configs[1]: batched paramgen.mlpg, %d utterances/GPU, T~U{%d..%d}, D=187 (mgc 180 + lf0 3 + vuv 1 "
                    "copied + bap 3), 3 windows, per-frame diagonal variances, float32 I/O" % (N_UTT, T_LO, T_HI),
        "utterances_per_gpu": N_UTT, "static_dims": 62, "windows": 3,
        "sharding": "single GPU (the --gpus N > 1 lines strong-scale configs[4]; see scale_workload)",
        "cache": "inputs (230 MB) + factor scratch (236 MB) per step exceed the 126 MB L2; no explicit flush",
    }


# ---- configs[4]: 8192 utterances, mixed T, strong scaling ---------------------------------------------
CFG5_UTT, CFG5_T_LO, CFG5_T_HI = 8192, 200, 2000


def cfg5_buckets(world):
    """Buckets per pass: enough that the last (exposed) transfer is a small part of the pass, few enough
    that a bucket still fills the GPU (>= 512 utterances = 1024 CTAs per launch): 8 / 8 / 4 / 2 at 1 / 2 / 4 / 8 ranks."""
    return max(2, min(8, CFG5_UTT // world // 512))


def cfg5_lengths():
    return np.random.default_rng(4242).integers(CFG5_T_LO, CFG5_T_HI + 1, size=CFG5_UTT).astype(np.int64)


def cfg5_utterance(u, T, device=None):
    """Synthetic (T, 187) means / variances of utterance u: the same numbers on whichever rank makes them."""
    import torch
    g = torch.Generator(device=device if device is not None else "cpu").manual_seed(777000 + int(u))
    m = torch.rand((int(T), D_IN), generator=g, device=device, dtype=torch.float32)
    v = torch.rand((int(T), D_IN), generator=g, device=device, dtype=torch.float32) + 0.1
    return m, v


def config_cfg5(n_gpus):
    return {
        "workload": "configs[4]: %d-utterance paramgen.mlpg batch, T~U{%d..%d} (9.0e6 frames), D=187 Merlin layout, 3 windows, "
                    "per-frame diagonal variances, float32 I/O, STRONG-scaled over %d GPU(s): ShardPlan (%d buckets, "
                    "longest-first greedy per bucket), inputs pre-sharded in HBM, per bucket solve -> in-place "
                    "all-gather (copy-engine pushes into IPC-shared peer buffers over NVLink; NNK_SHARD_TRANSPORT=nccl: NCCL "
                    "all_gather_into_tensor) overlapped with the next bucket; every rank ends with all trajectories"
                    % (CFG5_UTT, CFG5_T_LO, CFG5_T_HI, n_gpus, cfg5_buckets(n_gpus)),
        "utterances": CFG5_UTT, "static_dims": 62, "windows": 3, "buckets": cfg5_buckets(n_gpus),
        "sharding": "utterance-sharded, %d rank(s), %d bucketed all-gathers per pass (the path's only collective)"
                    % (n_gpus, cfg5_buckets(n_gpus)),
        "cache": "per-rank inputs (>= 1.7 GB) and factor scratch exceed the 126 MB L2; no explicit flush",
    }


# ---------------------------------------------------------------------------------------------------
# CPU reference arm
# ---------------------------------------------------------------------------------------------------
def make_cfg5_sample(n_sample=256):
    """Bounded CPU-arm sample of configs[4]: the first `n_sample` utterances of the 8192 (mixed T)."""
    lens = cfg5_lengths()[:n_sample]
    rng = np.random.default_rng(99)
    n = int(lens.sum())
    return lens, rng.random((n, D_IN), dtype=np.float32), rng.random((n, D_IN), dtype=np.float32) + np.float32(0.1)


def _ref_worker_init(workload="cfg2"):
    os.environ["OMP_NUM_THREADS"] = "1"
    global _BATCH
    # workers own the data: no pickling of 230 MB through pipes per step
    lens, m, v = make_cfg5_sample() if workload == "cfg5" else make_batch(0)
    _BATCH = (np.concatenate([[0], np.cumsum(lens)]), m, v)
    import warnings
    warnings.simplefilter("ignore")
    import oracle
    global _G
    if oracle.reference_available():
        oracle.import_reference()
        from nnmnkwii import paramgen as G_
        _G = G_.mlpg
    else:
        _G = oracle.mlpg


def _ref_one(u):
    off, m_all, v_all = _BATCH
    m, v = m_all[off[u]:off[u + 1]], v_all[off[u]:off[u + 1]]
    # the gallery-notebook pattern: per utterance, one paramgen.mlpg call per stream; vuv copied
    out = np.empty((m.shape[0], D_OUT), dtype=m.dtype)
    out[:, 0:60] = _G(m[:, 0:180], v[:, 0:180], WINDOWS)
    out[:, 60:61] = _G(m[:, 180:183], v[:, 180:183], WINDOWS)
    out[:, 61] = m[:, 183]
    out[:, 62:63] = _G(m[:, 184:187], v[:, 184:187], WINDOWS)
    return out.shape[0]


def usable_cores():
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:  # cgroup v2 CPU quota, if any
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(int(q) / int(per))))
    except Exception:
        pass
    return n


def cpu_reference(lens, means, variances, n_sample, repeats, cores=None, workload="cfg2"):
    """frames/s of the reference CPU path on `n_sample` utterances of the workload.  The reference is
    single-threaded; it is given one process per core, and because oversubscribed or throttled hosts
    make "all cores" slower than fewer, a few pool sizes are tried and the fastest is reported."""
    import multiprocessing as mp
    import oracle
    kind = "reference" if oracle.reference_available() else "port"
    off = np.concatenate([[0], np.cumsum(lens)])
    items = list(range(n_sample))
    frames = int(off[n_sample])
    # the reference is single-threaded by construction (.github/workflows/ci.yaml:17 pins OMP_NUM_THREADS=1);
    # one process per core, no BLAS/OpenMP thread pools inside the workers (the env is inherited on spawn)
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[var] = "1"
    ctx = mp.get_context("spawn")
    n_all = usable_cores()
    sizes = [cores] if cores else sorted({min(n_all, c) for c in (n_all, 64, 32, 16, 8)}, reverse=True)
    best = None
    tried = {}
    for size in sizes:
        with ctx.Pool(size, initializer=_ref_worker_init, initargs=(workload,)) as pool:
            pool.map(_ref_one, items[: max(size, 8)])  # warm-up (imports, page-in)
            times = []
            for _ in range(repeats):
                t0 = time.perf_counter()
                pool.map(_ref_one, items, chunksize=max(1, n_sample // (size * 4)))
                times.append(time.perf_counter() - t0)
        tried[size] = frames / min(times)
        if best is None or min(times) < min(best[1]):
            best = (size, times)
    size, times = best
    return {"value": frames / min(times), "unit": UNIT, "cores": size, "kind": kind,
            "sample": "%d of %d utterances (%d frames), per-utterance per-stream paramgen.mlpg, %d processes (of %d usable "
                      "cores; pool sizes tried -> frames/s: %s), best of %d"
                      % (n_sample, len(lens), frames, size, n_all, {k: round(v) for k, v in tried.items()}, repeats)}, times, frames


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # N > 1: our arm runs configs[4] (8192 ragged utterances); the CPU arm times a 256-utterance sample of it
    workload = "cfg5" if args.gpus > 1 else "cfg2"
    lens, means, variances = make_cfg5_sample() if workload == "cfg5" else make_batch(0)
    steps, warm = max(1, args.steps), max(0, args.warmup)
    # each step = one bounded sample of the workload (whole batch is ~1.5 CPU-seconds on one core)
    n_sample = len(lens)
    probe, _, _ = cpu_reference(lens, means, variances, n_sample, 3, workload=workload)  # best pool size (best of 3 each)
    base, times, frames = cpu_reference(lens, means, variances, n_sample, steps + warm, probe["cores"], workload=workload)
    base["sample"] = probe["sample"].rsplit(", best of", 1)[0] + ", %d timed steps" % steps
    timed = times[warm:] if len(times) > warm else times
    total = sum(timed)
    val = frames * len(timed) / total
    base["value"] = val
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": len(timed),
        "warmup": warm, "ms_per_step": 1e3 * total / len(timed), "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_cfg5(args.gpus) if workload == "cfg5" else config(args.gpus),
        "cpu_baseline": base,
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,utilization.gpu,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, smmax, reasons, busy = [], [], set(), []
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, mx, util = float(f[1]), float(f[2]), float(f[4])
            except ValueError:
                continue
            sm.append(clk); smmax.append(mx)
            if util > 0:
                busy.append(clk)
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        use = busy or sm
        return {"sm_mhz": statistics.median(use) if use else None, "sm_max_mhz": max(smmax) if smmax else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_under_load": len(busy)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profile_traffic(patterns):
    """DRAM bytes per launch of the dominant kernel, parsed from the newest committed ncu summary under
    profiles/ whose name matches `pattern` (dram__bytes_read.sum + dram__bytes_write.sum of one
    `ncu --set full` capture), so that the number in the JSON line and the profile cannot drift."""
    import glob
    import re
    files = []
    for pattern in patterns:  # first pattern with a match wins (newest round first)
        files = sorted(glob.glob(os.path.join(ROOT, "profiles", pattern)))
        if files:
            break
    for f in reversed(files):
        txt = open(f).read()
        got = {}
        for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            m = re.search(r"^%s\s+(\S+)\s+([0-9.eE+-]+)\s*$" % re.escape(key), txt, re.M)
            if m:
                unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(m.group(1))
                if unit:
                    got[key] = float(m.group(2)) * unit
        if len(got) == 2:
            return sum(got.values()), "profiles/%s (ncu --set full: dram__bytes_read.sum %.1f MB + dram__bytes_write.sum " \
                "%.1f MB per launch)" % (os.path.basename(f), got["dram__bytes_read.sum"] / 1e6, got["dram__bytes_write.sum"] / 1e6)
    return None, "no ncu --set full summary matching profiles/%s" % (patterns,)


class Cfg5Pass(object):
    """configs[4] resident on this rank in ShardPlan layout + one timed pass over it."""

    def __init__(self, rank, world, device, transport=None):
        import torch
        from nnmnkwii_b200 import paramgen as G
        from nnmnkwii_b200 import sharding
        self.rank, self.world, self.device = rank, world, device
        self.lens = cfg5_lengths()
        self.layout = G.merlin_layout()
        self.plan = sharding.ShardPlan(self.lens, world, cfg5_buckets(world))
        self.transport = transport if world > 1 else None
        self.batch = sharding.ShardedBatch(self.plan, rank, device, D_IN, D_OUT, torch.float32, transport=self.transport)
        for b in range(self.plan.n_buckets):  # inputs are generated straight into the rank's HBM slice
            for u in self.plan.members[b][rank]:
                m, v = cfg5_utterance(u, self.lens[u], device)
                l0 = int(self.plan.local_start[u])
                self.batch.means[l0:l0 + m.shape[0]] = m
                self.batch.variances[l0:l0 + m.shape[0]] = v
        self.status = torch.zeros(1, dtype=torch.int64, device=device)
        self.frames_local = self.plan.frames_of_rank(rank)
        self.frames_total = int(self.lens.sum())

    def run(self, group=None):
        from nnmnkwii_b200 import sharding
        sharding.solve_sharded(self.batch, WINDOWS, self.layout, group, status=self.status)

    def solve_only(self):
        from nnmnkwii_b200 import _device as dev
        from nnmnkwii_b200 import _lib
        from nnmnkwii_b200 import sharding
        wc = _lib.make_windows(WINDOWS)
        chains = dev.chains_on_device(self.layout.chains, self.device)
        for b in range(self.plan.n_buckets):
            sharding._solve_bucket(self.batch, b, wc, chains, self.layout.n_chain, self.status)

    def gather_only(self, group=None):
        """The collective alone (copy-engine pushes / NCCL), no solve running."""
        import torch
        from nnmnkwii_b200 import sharding
        if self.batch.peer is not None:
            cur = torch.cuda.current_stream(self.device)
            ev = torch.cuda.Event()
            ev.record(cur)
            for b in range(self.plan.n_buckets):
                n_rows = int(self.plan.lengths[self.plan.members[b][self.rank]].sum())
                self.batch.peer.push(self.plan.goff[b] + self.rank * self.plan.cap[b], n_rows, ev)
            self.batch.peer.finish(cur)
            return
        works = [sharding._gather_bucket(self.batch.result, self.plan, b, self.rank, group) for b in range(self.plan.n_buckets)]
        for w in works:
            if w is not None:
                w.wait()

    def parity(self, utts):
        """max relative error vs the oracle of the gathered trajectories of a few utterances (any owner)."""
        import oracle
        worst = 0.0
        for u in utts:
            m, v = cfg5_utterance(u, self.lens[u], self.device)
            m, v = m.cpu().numpy(), v.cpu().numpy()
            a = int(self.plan.row_start[u])
            got = self.batch.result[a:a + int(self.lens[u])].cpu().numpy()
            ref = oracle.mlpg(m[:, :180], v[:, :180], WINDOWS)
            worst = max(worst, float(np.abs(got[:, :60] - ref).max() / np.abs(ref).max()))
            assert np.array_equal(got[:, 61], m[:, 183])  # the copied vuv column
        return worst


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, **arrays):
    """--dump-outputs: each float32 / float64 array as out_dir/<name>.npy, DUMP_MAX_BYTES in all at most."""
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _timed(fn, steps, warmup, barrier):
    import torch
    for _ in range(warmup):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    return e0.elapsed_time(e1) / steps


def run_sharded(args, rank, world, local):
    """--gpus N > 1: configs[4] strong-scaled (see module docstring)."""
    import torch
    import torch.distributed as dist
    from nnmnkwii_b200 import _device as dev
    from nnmnkwii_b200 import _lib
    from nnmnkwii_b200 import paramgen as G

    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=device)
    from nnmnkwii_b200 import sharding
    transport = sharding.default_transport(device)
    job = Cfg5Pass(rank, world, device, transport)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    warm = max(3, args.warmup)
    sampler = ClockSampler(local)
    for _ in range(warm):
        job.run()
    barrier()
    dev.raise_if_failed(job.status)
    if rank == 0:
        sampler.start()
        time.sleep(0.2)
    n0 = _lib.launch_count()
    pass_ms = reduce_max(_timed(job.run, args.steps, 0, barrier))          # the metric: solve + gather, every step
    launches = _lib.launch_count() - n0
    clocks = sampler.stop() if rank == 0 else None
    kernel_ms = reduce_max(_timed(job.solve_only, max(3, args.steps // 2), 1, barrier))   # the solves alone (slowest rank)
    gather_ms = reduce_max(_timed(job.gather_only, max(3, args.steps // 2), 1, barrier))  # the 4 all-gathers alone
    value = job.frames_total / (pass_ms * 1e-3)
    parity = None
    if rank == 0:
        owners = {int(job.plan.owner[u]): u for u in range(CFG5_UTT - 1, -1, -1)}  # one utterance of every rank
        parity = job.parity(sorted(owners.values())[: min(world, 4)])

    # e2e at N GPUs: every rank pushes ITS shard through the public host-buffer API (pinned NumPy in,
    # NumPy out: H2D + solve + D2H every step); the trajectories land in host memory sharded the same way
    mine = np.concatenate([job.plan.members[b][rank] for b in range(job.plan.n_buckets)])
    lens_loc = job.lens[mine]
    rows = int(lens_loc.sum())
    hm = torch.empty((rows, D_IN), dtype=torch.float32).pin_memory()
    hv = torch.empty((rows, D_IN), dtype=torch.float32).pin_memory()
    o = 0
    for u in mine:
        a = int(job.plan.local_start[u])
        n = int(job.lens[u])
        hm[o:o + n].copy_(job.batch.means[a:a + n])
        hv[o:o + n].copy_(job.batch.variances[a:a + n])
        o += n
    hy = torch.empty((rows, D_OUT), dtype=torch.float32).pin_memory().numpy()
    hm, hv = hm.numpy(), hv.numpy()
    G.mlpg_batch(hm, hv, WINDOWS, lengths=lens_loc, layout=job.layout, out=hy)
    barrier()
    e2e_steps = 3
    n1 = _lib.launch_count()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        G.mlpg_batch(hm, hv, WINDOWS, lengths=lens_loc, layout=job.layout, out=hy)
    torch.cuda.synchronize()
    e2e_s = reduce_max(time.perf_counter() - t0)
    launches += _lib.launch_count() - n1
    e2e_val = job.frames_total * e2e_steps / e2e_s
    h2d = reduce_max(float(hm.nbytes + hv.nbytes))
    barrier()
    if job.batch.peer is not None:
        job.batch.peer.close()
    dist.barrier()
    dist.destroy_process_group()
    if rank != 0:
        return
    peak, peak_src = measured_peak()
    achieved = ALGO_BYTES_PER_FRAME * job.frames_local / (kernel_ms * 1e-3) / 1e9
    out_bytes = job.plan.rows_total * D_OUT * 4
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": pass_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config_cfg5(world),
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(rows * D_OUT * 4),
                "steps": e2e_steps, "api": "per rank: nnmnkwii_b200.paramgen.mlpg_batch(numpy pinned, its shard of configs[4]) -> "
                "nnk_mlpg_batch_host; bytes are per rank (largest shard); no gather: results stay sharded in host memory"},
        "gpu_launches": int(launches),
        "kernel_ms": kernel_ms, "allgather_ms": gather_ms, "allgather_exposed_ms": max(0.0, pass_ms - kernel_ms),
        "kernel_plus_allgather_ms": kernel_ms + gather_ms,
        "allgather": {"transport": transport, "bytes_received_per_rank": int(out_bytes * (world - 1) / world), "buckets": job.plan.n_buckets,
                      "alone_gbs_per_rank": out_bytes * (world - 1) / world / (gather_ms * 1e-3) / 1e9,
                      "note": "every rank must RECEIVE (N-1)/N of the 2.27 GB result per pass: at N=8 that is 1.98 GB over one "
                              "NVLink port (<= 900 GB/s/dir) >= 2.2 ms against ~1.05 ms of solve -- the pass is NVLink-receive "
                              "bound, which no overlap can hide; the solves alone scale as kernel_ms shows"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None, "peak_source": peak_src, "kernel": "mlpg_fwd_as_kernel (per rank, %d bucket launches)" % job.plan.n_buckets,
                     "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": ALGO_BYTES_PER_FRAME * job.frames_local},
        "cpu_baseline": None, "clocks": clocks, "parity_max_rel_err_vs_oracle": parity,
        "frames_per_step_per_gpu": job.frames_local, "frames_per_step": job.frames_total,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node == --gpus"
    if world > 1:
        return run_sharded(args, rank, world, local)
    lens, means, variances = make_batch(rank)

    # CPU baseline first (rank 0, before CUDA is touched in this process; spawn-based pool)
    cpu_base = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu_base, _, _ = cpu_reference(lens, means, variances, N_UTT, 2)

    torch.cuda.set_device(local)
    device = torch.device("cuda", local)

    from nnmnkwii_b200 import _device as dev
    from nnmnkwii_b200 import _lib
    from nnmnkwii_b200 import paramgen as G

    layout = G.merlin_layout()
    n_rows = int(lens.sum())
    off_np = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    wc = _lib.make_windows(WINDOWS)

    # ---- device-resident arm --------------------------------------------------------------------
    d_m = torch.from_numpy(means).to(device)
    d_v = torch.from_numpy(variances).to(device)
    d_out = torch.zeros((n_rows, D_OUT), dtype=torch.float32, device=device)
    d_off = torch.from_numpy(off_np).to(device)
    d_order = torch.from_numpy(np.argsort(-lens, kind="stable").astype(np.int32)).to(device)
    d_chains = dev.chains_on_device(layout.chains, device)
    max_T = int(lens.max())

    d_status = torch.zeros(1, dtype=torch.int64, device=device)  # caller-owned status word: keeps the first failure

    def step():  # one launch of the solve kernel and nothing else (scratch comes from the caching allocator)
        return dev.run_mlpg("fwd", means=d_m, variances=d_v, rhs=None, out=d_out, offsets=d_off, lengths=None,
                            order=d_order, chains=d_chains, n_chain=layout.n_chain, max_T=max_T, windows_c=wc,
                            in_ld=D_IN, var_ld=D_IN, go_ld=0, out_ld=D_OUT, dtype_code=_lib.NNK_F32, go_f64=0,
                            n_utt=N_UTT, device=device, check=False, status=d_status)

    for _ in range(max(3, args.warmup)):
        status = step()
    torch.cuda.synchronize()
    dev.raise_if_failed(status)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.2)

    def barrier():
        torch.cuda.synchronize()

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    n0 = _lib.launch_count()
    barrier()
    ev0.record()
    for i in range(args.steps):
        kev[i][0].record()
        step()
        kev[i][1].record()
    ev1.record()
    barrier()
    launches = _lib.launch_count() - n0
    total_ms = ev0.elapsed_time(ev1)
    kernel_ms = [a.elapsed_time(b) for a, b in kev]
    frames_all = float(n_rows)
    value = frames_all * args.steps / (total_ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, trajectories=d_out.cpu().numpy())

    # parity spot check of what was just timed (utterance 0, mgc stream) against the oracle
    parity = None
    if rank == 0:
        import oracle
        a, b = int(off_np[0]), int(off_np[1])
        ref = oracle.mlpg(means[a:b, :180], variances[a:b, :180], WINDOWS)
        got = d_out[a:b, :60].cpu().numpy()
        parity = float(np.abs(got - ref).max() / np.abs(ref).max())

    # ---- end-to-end arm: public API on pinned host buffers ------------------------------------------
    e2e_steps = max(3, min(args.steps, args.e2e_steps))
    pm = torch.from_numpy(means).pin_memory()
    pv = torch.from_numpy(variances).pin_memory()
    hm, hv = pm.numpy(), pv.numpy()
    hy = torch.empty((n_rows, D_OUT), dtype=torch.float32).pin_memory().numpy()
    for _ in range(2):
        y = G.mlpg_batch(hm, hv, WINDOWS, lengths=lens, layout=layout, out=hy)
    barrier()
    n1 = _lib.launch_count()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        y = G.mlpg_batch(hm, hv, WINDOWS, lengths=lens, layout=layout, out=hy)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    launches += _lib.launch_count() - n1
    e2e_val = frames_all * e2e_steps / e2e_s
    if rank == 0:
        assert np.array_equal(y[: int(off_np[1])], d_out[: int(off_np[1])].cpu().numpy()), "e2e and device paths disagree"

    clocks = sampler.stop()  # the clocks of the timed region (+ the e2e arm), not of the side measurements
    extras = dtw = scale = None
    if not args.no_extras:
        try:
            extras = bench_extras(device)
            dtw = extras.pop("dtw", None)
        except Exception as e:  # the headline line must survive a failure of the side measurements
            extras = {"error": repr(e)}
        try:
            scale = bench_cfg5_single(device, max(3, min(10, args.steps)))
        except Exception as e:
            scale = {"error": repr(e)}
    peak, peak_src = measured_peak()
    traffic, traffic_src = profile_traffic(DOMINANT_PROFILES)
    k_ms = statistics.mean(kernel_ms)
    achieved = ALGO_BYTES_PER_FRAME * n_rows / (k_ms * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "strong",  # the --gpus N > 1 lines strong-scale configs[4]; its one-GPU pass is `scale_workload` below
        "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config(world),
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(means.nbytes + variances.nbytes),
                "d2h_bytes_per_step": int(n_rows * D_OUT * 4), "steps": e2e_steps,
                "api": "nnmnkwii_b200.paramgen.mlpg_batch(numpy pinned) -> nnk_mlpg_batch_host"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src + "; the excess over the algorithmic bytes is the "
                     "float64 factor scratch round trip", "peak_source": peak_src, "kernel": ("mlpg_kernel<float,3,1,1,FWD> (register prefetch)" if os.environ.get("NNK_MLPG_DIRECT") == "1" else
                                "mlpg_fwd_tma_kernel<float,3,1,1,STD> (single warp)" if os.environ.get("NNK_MLPG_SINGLE") == "1" else
                                "mlpg_fwd_as_kernel<float,3,1,1,STD> (3 assembler warps + 1 solver warp per 32 chains)"),
                     "kernel_ms": k_ms, "algorithmic_bytes_per_launch": ALGO_BYTES_PER_FRAME * n_rows},
        "cpu_baseline": cpu_base,
        "clocks": clocks,
        "parity_max_rel_err_vs_oracle": parity,
        "frames_per_step_per_gpu": n_rows,
        "dtw": dtw,
        "scale_workload": scale,
        "other_kernels": extras,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
# the other kernels of the path (reported as extra keys next to the headline metric)
# ---------------------------------------------------------------------------------------------------
def make_dtw_pairs(n_pairs, seed=4321):
    """configs[3]: random MFCC-like 25-dim pairs, T~U{700..900}; Y = monotone time-warp of X + noise."""
    rng = np.random.default_rng(seed)
    D, Tmax = 25, 900
    X = np.zeros((n_pairs, Tmax, D), np.float32)
    Y = np.zeros((n_pairs, Tmax, D), np.float32)
    for n in range(n_pairs):
        Tx, Ty = int(rng.integers(700, 901)), int(rng.integers(700, 901))
        x = (np.cumsum(rng.standard_normal((Tx, D)), 0) * 0.1).astype(np.float32)
        src = np.sort(rng.random(Ty)) * (Tx - 1)
        y = x[np.round(src).astype(int)] + 0.05 * rng.standard_normal((Ty, D)).astype(np.float32)
        X[n, :Tx], Y[n, :Ty] = x, y
    return X, Y


def _device_ms(fn, reps):
    """Average device time of fn(): `reps` calls captured into one CUDA graph and replayed (so that the
    host-side cost of issuing short kernels from Python is not what gets measured); eager timing if the
    calls cannot be captured."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    try:
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(reps):
                fn()
        graph.replay()
        torch.cuda.synchronize()
        e0.record()
        graph.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps, "cuda_graph"
    except Exception:
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps, "eager"


def _dtw_cpu_one(args):
    import oracle
    x, y, radius = args
    return oracle.fastdtw(x, y, radius=radius, kind="melcd")[3]


def dtw_cpu_baseline(X, Y, n_c=64, n_py=16):
    """CPU numbers beside the DTW kernels (BASELINE.md 3.4): OUR restatement, not the fastdtw package
    (absent, unpinned: setup.py:139).  (i) the C oracle -- exact O(Tx*Ty) DP and FastDTW(radius=1), float64,
    same 3-way min / tie order -- one process per host core on `n_c` pairs; (ii) the faithful pure-Python
    FastDTW with a per-cell Python callback (what a user of the reference experiences) on `n_py` pairs, 1 core."""
    import multiprocessing as mp
    import oracle
    from oracle import fastdtw_py
    lens = lambda A, n: int(np.flatnonzero(np.abs(A[n]).sum(1) >= 1e-7)[-1] + 1)
    pairs = [(X[n, :lens(X, n)], Y[n, :lens(Y, n)]) for n in range(len(X))]
    n_c, n_py = min(n_c, len(pairs)), min(n_py, len(pairs))
    cores = min(usable_cores(), n_c)
    out = {"kind": "port", "label": "restated oracle, not fastdtw", "cores": cores,
           "sample": "C oracle: all %d pairs FastDTW(radius=1), %d pairs exact DP (%d processes); per-cell-callback Python "
                     "FastDTW: %d pairs (1 core)" % (len(pairs), n_c, cores, n_py)}
    with mp.get_context("spawn").Pool(cores) as pool:
        pool.map(_dtw_cpu_one, [(p[0][:50], p[1][:50], 1) for p in pairs[:cores]])  # warm-up: imports, library load
        for name, radius in (("fastdtw_radius1", 1), ("exact", -1)):
            t0 = time.perf_counter()
            sub = pairs if radius > 0 else pairs[:n_c]
            cells = sum(pool.map(_dtw_cpu_one, [(p[0], p[1], radius) for p in sub], chunksize=1))
            out[name + "_c_oracle"] = {"value": cells / (time.perf_counter() - t0), "unit": "cell-updates/s", "cores": cores}
    t0 = time.perf_counter()
    cells = 0
    for x, y in pairs[:n_py]:
        cells += fastdtw_py.fastdtw(x, y, radius=1, dist=lambda a, b: oracle.LOGDB_CONST * np.sqrt(((a - b) ** 2).sum()),
                                    return_cells=True)[2]
    out["fastdtw_radius1_python_callback"] = {"value": cells / (time.perf_counter() - t0), "unit": "cell-updates/s", "cores": 1}
    return out


def bench_cfg5_single(device, steps):
    """configs[4] on ONE GPU, measured like the N>1 arm (same plan, buckets, kernels; no collective): the
    denominator of the scaling efficiency of the --gpus N lines."""
    import torch
    job = Cfg5Pass(0, 1, device)
    ms = _timed(job.solve_only, steps, 2, torch.cuda.synchronize)
    from nnmnkwii_b200 import _device as dev
    dev.raise_if_failed(job.status)
    worst = job.parity([0, CFG5_UTT - 1])
    peak, _ = measured_peak()
    gbs = ALGO_BYTES_PER_FRAME * job.frames_total / (ms * 1e-3) / 1e9
    return {"workload": config_cfg5(1)["workload"], "value": job.frames_total / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
            "steps": steps, "frames_per_step": job.frames_total, "hbm_gbs_algorithmic": gbs, "roofline_frac": gbs / peak,
            "parity_max_rel_err_vs_oracle": worst}


def bench_extras(device, reps=5):
    import torch
    from nnmnkwii_b200 import autograd as AF
    from nnmnkwii_b200 import paramgen as G
    from nnmnkwii_b200.preprocessing import alignment as A
    out = {}
    # --- DTW, configs[3]: 512 pairs, melcd cost; cell updates/s next to the CPU restatement ------------------
    X, Y = make_dtw_pairs(512)
    Xd, Yd = torch.from_numpy(X).to(device), torch.from_numpy(Y).to(device)
    dtw = {"workload": "configs[3]: 512 pairs, T~U{700..900}, 25-dim, melcd local cost; trim + DTW per batch (no gather)",
           "unit": "cell-updates/s", "parity": "paths, cell counts and distance bit-identical to the restated oracle "
           "(tests/test_dtw_gpu.py); the real fastdtw package is absent: parity unpinned"}
    for name, radius in (("fastdtw_radius1", 1), ("exact", -1)):
        res = A._align_batch(Xd, Yd, 1, radius)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            res = A._align_batch(Xd, Yd, 1, radius)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        cells = int(res.cells.sum().item())
        dtw[name] = {"value": cells / (ms * 1e-3), "cells_per_batch": cells, "pairs": 512, "ms_per_batch": ms}
    dtw["cpu_baseline"] = dtw_cpu_baseline(X, Y)
    out["dtw"] = dtw
    # --- UnitVarianceMLPG fwd + loss.backward(), configs[2] ---------------------------------------------
    T, sd, B = 1000, 60, 64
    R = torch.from_numpy(G.unit_variance_mlpg_matrix(WINDOWS, T)).to(device)
    g = torch.Generator(device=device).manual_seed(0)
    mu = torch.randn(B, T, 3 * sd, device=device, generator=g).requires_grad_(True)
    for _ in range(2):
        AF.unit_variance_mlpg(R, mu).pow(2).mean().backward()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        mu.grad = None
        AF.unit_variance_mlpg(R, mu).pow(2).mean().backward()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    out["unit_variance_mlpg_fwd_bwd"] = {"frames_per_sec": B * T / (ms * 1e-3), "ms_per_iter": ms, "batch": B, "T": T,
                                         "static_dim": sd,
                                         "includes": "autograd step: stencil fwd + loss (torch) + stencil bwd + Python/launch overhead"}
    try:  # the same step captured once and replayed as a CUDA graph: what is left when the Python / dispatch cost is gone
        go_s = torch.ones(B, T, sd, device=device)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                yy = AF.unit_variance_mlpg(R, mu)
                (gg,) = torch.autograd.grad(yy, mu, go_s)
        torch.cuda.current_stream().wait_stream(side)
        graph.replay()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(20):
            graph.replay()
        e1.record()
        torch.cuda.synchronize()
        out["unit_variance_mlpg_fwd_bwd"]["ms_per_iter_cuda_graph"] = e0.elapsed_time(e1) / 20
        out["unit_variance_mlpg_fwd_bwd"]["cuda_graph_includes"] = "fwd sweep + bwd sweep (grad_output given), one graph replay"
    except Exception as e:
        out["unit_variance_mlpg_fwd_bwd"]["cuda_graph_error"] = repr(e)
    # the two stencil sweeps alone (device time of the C-ABI calls, CUDA events)
    from nnmnkwii_b200 import _uvmlpg as uv
    band = uv.band_of(R, device)
    # rotate over 4 input sets (4 x 61 MB > the 126 MB L2) so that the sweeps stream from HBM
    xs = [torch.randn(B, T, 3 * sd, device=device, generator=g) for _ in range(4)]
    gos = [torch.randn(B, T, sd, device=device, generator=g) for _ in range(8)]
    turn = [0]

    def fwd_call():
        turn[0] += 1
        return uv.apply_forward(band, xs[turn[0] % 4], False)

    def bwd_call():
        turn[0] += 1
        return uv.apply_backward(band, gos[turn[0] % 8], False, 3 * sd)
    for name, fn in (("fwd", fwd_call), ("bwd", bwd_call)):
        ms, how = _device_ms(fn, 20)
        out["unit_variance_mlpg_" + name + "_sweep"] = {"ms": ms, "timing": how, "algorithmic_bytes": 61.44e6, "hbm_gbs_algorithmic": 61.44e6 / (ms * 1e-3) / 1e9,
                                                       "band_half_width": band.K, "toeplitz_rows": (band.toep[1] - band.toep[0]) if band.toep else 0}
    # --- MLPG at the north_star shape: T=1000, static_dim=60, 3 windows; fwd and mlpg_grad --------------
    from nnmnkwii_b200 import _device as dev
    from nnmnkwii_b200 import _lib
    B2, T2, sd2 = 256, 1000, 60
    wc = _lib.make_windows(WINDOWS)
    chains = dev.chains_on_device(dev.simple_chains(sd2), device)
    off = torch.arange(B2 + 1, dtype=torch.int64, device=device) * T2
    m2 = torch.rand(B2 * T2, 3 * sd2, device=device, generator=g)
    v2 = torch.rand(B2 * T2, 3 * sd2, device=device, generator=g) + 0.1
    v1 = torch.rand(3 * sd2, device=device, generator=g) + 0.1
    go2 = torch.randn(B2 * T2, sd2, device=device, generator=g)
    y2 = torch.zeros(B2 * T2, sd2, device=device)
    g2 = torch.zeros(B2 * T2, 3 * sd2, device=device)

    def run(mode, var, var_ld, rhs, o, out_ld):
        return dev.run_mlpg(mode, means=m2, variances=var, rhs=rhs, out=o, offsets=off, lengths=None, order=None,
                            chains=chains, n_chain=sd2, max_T=T2, windows_c=wc, in_ld=3 * sd2, var_ld=var_ld,
                            go_ld=sd2, out_ld=out_ld, dtype_code=_lib.NNK_F32, go_f64=0, n_utt=B2, device=device,
                            check=False)
    cases = (("mlpg_fwd_T1000_sd60", lambda: run("fwd", v2, 3 * sd2, None, y2, sd2), 28 * sd2),
             ("mlpg_fwd_T1000_sd60_global_variance", lambda: run("fwd", v1, 0, None, y2, sd2), 16 * sd2),
             ("mlpg_grad_T1000_sd60", lambda: run("grad", v2, 3 * sd2, go2, g2, 3 * sd2), 28 * sd2))
    for name, fn, bytes_per_frame in cases:
        ms, how = _device_ms(fn, 10)
        out[name] = {"frames_per_sec": B2 * T2 / (ms * 1e-3), "ms": ms, "timing": how, "utterances": B2,
                     "hbm_gbs_algorithmic": bytes_per_frame * B2 * T2 / (ms * 1e-3) / 1e9}
    # --- masked melcd over aligned-output sized batches (SURVEY 8f row 4) --------------------------------
    import ctypes
    Bm, Tm, Dm = 2048, 1600, 25  # 2 x 328 MB: larger than L2, long enough that launch overhead is noise
    Xm = torch.randn(Bm, Tm, Dm, device=device, generator=g)
    Ym = torch.randn(Bm, Tm, Dm, device=device, generator=g)
    lens_m = torch.randint(700, Tm + 1, (Bm,), generator=torch.Generator().manual_seed(5)).to(device=device, dtype=torch.int32)
    need = int(_lib.lib.nnk_metric_workspace_bytes(Bm, Tm))
    wsm = torch.zeros(need, dtype=torch.uint8, device=device)
    res = torch.zeros(2, dtype=torch.float64, device=device)
    def melcd_call():
        _lib.check(_lib.lib.nnk_frame_metric(Xm.data_ptr(), Ym.data_ptr(), _lib.NNK_F32, Bm, Tm, Dm, Tm * Dm, Dm,
                                             lens_m.data_ptr(), 0, ctypes.c_void_p(res.data_ptr()),
                                             ctypes.c_void_p(res.data_ptr() + 8), ctypes.c_void_p(wsm.data_ptr()),
                                             ctypes.c_int64(need), dev.current_stream_ptr(device)), "nnk_frame_metric")
    ms, how = _device_ms(melcd_call, 20)
    nbytes = 2 * 4 * Dm * int(lens_m.sum().item())
    out["masked_melcd"] = {"ms": ms, "frames": int(lens_m.sum().item()), "algorithmic_bytes": nbytes,
                           "hbm_gbs_algorithmic": nbytes / (ms * 1e-3) / 1e9, "timing": how, "includes": "one reduction kernel launch per call"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, save the trajectories of the last step as DIR/trajectories.npy "
                         "(all utterances in batch order, (frames, 63) float32) for output-for-output comparison of builds")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs applies to the one-GPU run of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
