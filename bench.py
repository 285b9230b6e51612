#!/usr/bin/env python
"""bench.py -- throughput of the quorum-tally + Reed-Solomon accept path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3|cfg2|cfg3b|cfg4|cfg5]
                  [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input.  Default workload (cfg3,
BASELINE.json configs[2], the configuration the north-star target is quoted on): the fused RSPaxos accept
step -- RS(3,2) encode of 2^20 groups' 4096-byte request batches + quorum tally (4 of 5) of each group's
64-slot ack window -- ONE kernel launch per step, inputs resident in HBM.  The same JSON line carries the other
BASELINE configs as sub-benches: "cfg2" (MultiPaxos tally), "cfg3b" (reconstruct), "cfg4" (Crossword ragged
encode + distribute + coverage tally) and "cfg5" (Raft scan), each with its own roofline object.

  value      RS shard GB/s = (d+p)*L bytes per codeword * codewords / time   (whole job, all ranks)
  e2e        same metric through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside)
  roofline   algorithmic bytes per launch / CUDA-event kernel time vs MEASURED_PEAKS.json hbm_gbs
  cpu_baseline / --impl reference: the CPU oracle port of the reference path on this box's cores

N > 1 (one process per GPU): groups shard across ranks; replica r of a group led from rank h is simulated on rank
(h + r) % N, the encode kernel stores shard r there over NVLink and step flags in device memory order the followers'
acks and the next tally (summerset_b200/replicate.py) -- no host synchronisation, NCCL call or memcpy between steps.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# The CPU arm's OpenMP team is pinned one thread per physical core; libgomp reads these when it is first loaded and
# then also binds the INITIAL thread to the first place, so they are set only in the process that runs the CPU arm
# (--impl reference; the GPU arm's cpu_baseline leg runs that in a subprocess).  torchrun's OMP_NUM_THREADS=1 does not
# matter: thread counts are passed explicitly.
FULL_AFFINITY = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
if "reference" in sys.argv:
    os.environ.setdefault("OMP_PROC_BIND", os.environ.get("SS_CPU_BIND", "close"))
    os.environ.setdefault("OMP_PLACES", "cores")

import numpy as np  # noqa: E402

D, P, DATA_LEN = 3, 2, 4096
R, THRESH_RSPAXOS, THRESH_MULTIPAXOS = 5, 4, 3
G_PER_GPU = 1 << 20
METRIC = "RS shard GB/s on the fused RSPaxos accept step (RS(3,2) encode + quorum tally); consensus slots committed/s in slots_committed_per_s"
NVLINK_REF_GBS = 770.0      # measured peer copy per direction, B200_PROFILING.md


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg3", "cfg2", "cfg5", "cfg3b", "cfg4"])
    ap.add_argument("--groups", type=int, default=G_PER_GPU, help="groups per GPU")
    ap.add_argument("--variant", type=int, default=0, help="encode kernel variant (tuning)")
    ap.add_argument("--replicas", type=int, default=5, help="cfg3 variant: population n (RS(majority, n-majority), f=(n//2)//2)")
    ap.add_argument("--rs", default="", help="cfg3 variant: an arbitrary code 'd,p' (n = d+p replicas), e.g. 6,4 -- codes without a "
                                             "compile-time table are specialised at run time by NVRTC (variant bit 17 turns that off)")
    ap.add_argument("--exchange", default="ce", choices=["ce", "p2p", "nccl"],
                    help="N>1: how shard planes reach the simulated peers: ce = encode into local staging + copy-engine push overlapped "
                         "with the next step's encode; p2p = the encode kernel stores into the peers' HBM itself; nccl = all-to-all baseline")
    ap.add_argument("--lag", type=int, default=2, choices=[1, 2], help="N>1: the tally of step k reads the acks of step k-lag")
    ap.add_argument("--timeline", default="", help="N>1: write per-rank per-step CUDA-event timings to this JSON file")
    ap.add_argument("--no-tally", action="store_true", help="tuning: time the encode alone")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the cfg2/cfg3b/cfg4/cfg5 sub-benches")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="cfg3 / cfg2: after the timed steps, write what the last timed step computed (a seeded sample of the "
                         "groups: parity planes, commit words, commit_bar) to DIR/<name>.npy, so that two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in ("cfg3", "cfg2")):
        ap.error("--dump-outputs covers the GPU arm's cfg3 and cfg2 steps")
    return args


def measured_peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        j = json.loads(f.read_text())
        return float(j["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def copy_bandwidth_here(torch, dev):
    """STREAM-style copy on THIS box, measured the way MEASURED_PEAKS.json was (b.copy_(a), 1 Gi bf16 elements,
    read+write bytes, best of 10): boxes of the pool differ by several percent, so the live figure is reported
    beside the pool-wide denominator."""
    try:
        a = torch.empty(1 << 30, dtype=torch.bfloat16, device=dev)
        b = torch.empty_like(a)
        a.fill_(1.0)
        best = 0.0
        for _ in range(10):
            s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
            s.record(); b.copy_(a); e.record(); torch.cuda.synchronize()
            best = max(best, 2 * a.numel() * 2 / (s.elapsed_time(e) * 1e-3) / 1e9)
        del a, b
        return best
    except Exception:
        return None


def profile_traffic(key: str):
    """dram bytes per launch from the committed ncu --set full captures (profiles/traffic.json), or None."""
    f = ROOT / "profiles" / "traffic.json"
    if f.exists():
        try:
            return json.loads(f.read_text()).get(key)
        except Exception:
            return None
    return None


def roofline_obj(alg_bytes, ms, peak, peak_src, kernel, traffic_key, **extra):
    ach = alg_bytes / (ms * 1e-3) / 1e9
    d = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
         "traffic": profile_traffic(traffic_key), "kernel": kernel, "kernel_ms": ms,
         "algorithmic_bytes_per_launch": int(alg_bytes), "peak_source": peak_src + " (burst figure; kernel timed alone)"}
    d.update(extra)
    return d


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nme, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# =================================================================================================
# host topology helpers
# =================================================================================================
def physical_cores(cpus):
    """Number of distinct physical cores among `cpus` (SMT siblings counted once), from sysfs."""
    seen = set()
    for c in cpus:
        try:
            sib = Path(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read_text().strip()
        except Exception:
            sib = str(c)
        seen.add(sib)
    return max(1, len(seen))


def gpu_numa_cpus(torch, index: int):
    """CPUs of the NUMA node the GPU hangs off (sysfs), or None."""
    try:
        props = torch.cuda.get_device_properties(index)
        bus = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text().strip())
        if node < 0:
            return None, None
        txt = Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip()
        cpus = set()
        for part in txt.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        return node, cpus
    except Exception:
        return None, None


class NumaPin:
    """Runs a block with the process bound to the GPU's NUMA node, so that pinned host buffers allocated (first
    touched) inside it are local to the GPU's PCIe root and the copy-issuing thread runs next to them."""

    def __init__(self, torch, index: int):
        self.node, cpus = gpu_numa_cpus(torch, index)
        self.saved = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
        self.cpus = (cpus & FULL_AFFINITY) if (cpus and FULL_AFFINITY) else None

    def __enter__(self):
        if self.cpus:
            try:
                os.sched_setaffinity(0, self.cpus)
            except Exception:
                self.cpus = None
        return self

    def __exit__(self, *a):
        if self.cpus and self.saved:
            os.sched_setaffinity(0, self.saved)


# =================================================================================================
# CPU arm: the oracle port of the reference path on the box's host cores
# =================================================================================================
def cpu_arm(steps: int, warmup: int, n_cw: int, workload: str):
    """Times the C restatement of the reference path (oracle/ss_oracle.c: AVX2 vpshufb nibble tables -- what the
    crate's simd-accel feature gives -- OpenMP over codewords) on the WHOLE workload of one GPU.  Stable by
    construction: one thread per physical core (OMP_PLACES=cores, OMP_PROC_BIND=close), a static partition of the
    codewords, and every input / output page first touched by the thread that later encodes it."""
    from oracle import pyoracle as oracle
    cpus = sorted(FULL_AFFINITY) if FULL_AFFINITY else list(range(os.cpu_count() or 1))
    threads = physical_cores(cpus)
    if os.environ.get("SS_CPU_THREADS"):                 # tuning knobs (profiles/r02_cpu_arm_sweep.txt)
        threads = int(os.environ["SS_CPU_THREADS"])
    mode = (1 if oracle.have_avx2() else 0) | (0 if os.environ.get("SS_CPU_SCHED") == "dynamic" else oracle.MODE_STATIC)
    L = oracle.cw_shard_len(DATA_LEN, D)
    ds = (L + 15) // 16 * 16
    stride = (DATA_LEN + 15) // 16 * 16
    thr = THRESH_RSPAXOS if workload != "cfg2" else THRESH_MULTIPAXOS
    data = np.empty(n_cw * stride, dtype=np.uint8)
    oracle.first_touch_fill(data, n_cw, stride, stride, 0x5EED0003, False, threads)
    parity = np.empty(P * n_cw * ds, dtype=np.uint8)
    for j in range(P):
        oracle.first_touch_fill(parity[j * n_cw * ds:], n_cw, ds, ds, 0, True, threads)
    planes = np.empty(R * n_cw, dtype=np.uint64)
    for r in range(R):
        oracle.first_touch_fill(planes[r * n_cw:(r + 1) * n_cw].view(np.uint8), n_cw, 8, 8, 0xACC0 + r, False, threads)
    planes = planes.reshape(R, n_cw)
    planes[0] = np.uint64(0xFFFFFFFFFFFFFFFF)
    off = np.arange(n_cw, dtype=np.uint64) * np.uint64(stride)
    lens = np.full(n_cw, DATA_LEN, dtype=np.uint32)
    poff = np.arange(n_cw, dtype=np.uint64) * np.uint64(ds)

    def step():
        if workload != "cfg2":
            oracle.rs_encode_batch(D, P, data, off, lens, parity, n_cw * ds, poff, mode, threads)
        oracle.tally_planes(planes, thr, threads)

    for _ in range(max(1, warmup)):
        step()
    times = []
    for _ in range(max(1, steps)):
        t0 = time.perf_counter(); step(); times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    gbs = lambda dt: (D + P) * L * n_cw / dt / 1e9
    return dict(ms_per_step=med * 1e3, gbs=gbs(med), gbs_min=gbs(max(times)), gbs_max=gbs(min(times)),
                slots_per_s=n_cw * 64 / med, threads=threads, hw_threads=len(cpus), steps=len(times),
                path=("AVX2 vpshufb nibble tables (what rse-simd enables)" if (mode & 1) else "scalar MUL_TABLE")
                     + ", OpenMP static partition, 1 thread per physical core, NUMA first-touch",
                sample=f"{n_cw} codewords x {DATA_LEN} B (the whole per-GPU workload) + their 64-slot ack windows per step; "
                       f"median of {len(times)} steps")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_arm(args.steps, max(1, args.warmup), args.groups, args.workload)
    value = r["gbs"] if args.workload != "cfg2" else r["slots_per_s"]
    unit = "GB/s" if args.workload != "cfg2" else "slots/s"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": unit, "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": max(1, args.warmup), "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": config_dict(args, 1),
        "slots_committed_per_s": r["slots_per_s"],
        "cpu_baseline": {"value": value, "unit": unit, "cores": r["threads"], "hw_threads": r["hw_threads"], "kind": "port",
                         "sample": r["sample"], "path": r["path"], "min": r["gbs_min"], "max": r["gbs_max"],
                         "note": "C restatement of the reference's Rust path (oracle/ss_oracle.c); the reference itself cannot "
                                 "be built here (no cargo/rustc).  One host, so the workload is ONE GPU's share (groups x1) at "
                                 "every --gpus N"},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


WORKLOAD_TEXT = {
    "cfg3": "cfg3: RSPaxos (3,5) fused RS(3,2) encode + quorum tally (4 of 5), 2^20 groups x 4096 B request batch + 64-slot ack window per GPU",
    "cfg2": "cfg2: MultiPaxos 5-replica quorum tally (3 of 5), 2^20 groups x 64 slots per GPU",
    "cfg3b": "cfg3b: reconstruct_data, 2^20 codewords, 50% intact / 25% one data shard / 25% two shards missing",
    "cfg4": "cfg4: Crossword n=5 d=3 T=5 f=2, 2^20 codewords, data_len uniform over {256..65536}, spr uniform {1,2,3}",
    "cfg5": "cfg5: Raft 7-replica match-index commit scan, 2^22 groups, 64-slot term window",
}


def config_dict(args, world):
    L = (DATA_LEN + D - 1) // D
    txt = WORKLOAD_TEXT[args.workload]
    if args.workload == "cfg3" and (R != 5 or D != 3):
        txt = f"cfg3 variant: RSPaxos ({D},{R}) fused RS({D},{P}) encode + quorum tally ({THRESH_RSPAXOS} of {R}), 2^20 groups x 4096 B per GPU"
    return {"workload": txt,
            "groups_per_gpu": args.groups, "data_len": DATA_LEN, "rs": [D, P], "shard_len": L, "replicas": R,
            "sharding": f"groups x{world} (independent shards)" + ("" if world == 1 else
                        f" + shard planes delivered to the simulated peers' GPUs over NVLink (exchange = {args.exchange}); followers' ack planes "
                        "stored back by a follower kernel; ordering by step flags in device memory (no host sync or NCCL per step)"),
            "l2": "inputs (4 GiB payload + 2.9 GB parity per GPU) exceed the 126 MB L2; no flush needed"}


def _time_steps(torch, fn, steps, warmup):
    for _ in range(max(3, warmup)):
        fn()
    torch.cuda.synchronize()
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


DUMP_BYTES = 60_000_000     # --dump-outputs stays under 64 MB
DUMP_SEED = 0x5EED0D


def dump_step_outputs(torch, dev, out_dir, parity, committed, bar, n, L):
    """Writes what one accept step returned, for a fixed seeded sample of its n groups, as float arrays:
    groups (the sampled group indices), parity (P, k, L) shard bytes, commit_words (k, 2) low / high 32 bits of each
    commit bitmap, commit_bar (k,).  parity is None when the step did not encode, committed / bar when it did not tally."""
    per_group = (parity.shape[0] * L * 4 if parity is not None else 0) + (24 if committed is not None else 0) + 8
    k = min(n, DUMP_BYTES // per_group)
    idx = np.arange(n) if k == n else np.sort(np.random.default_rng(DUMP_SEED).choice(n, k, replace=False))
    idx_t = torch.from_numpy(idx).to(dev)
    out = {"groups": idx.astype(np.float64)}
    if parity is not None:
        out["parity"] = parity[:, idx_t, :L].cpu().numpy().astype(np.float32)
    if committed is not None:
        cw = committed[idx_t].cpu().numpy().view(np.uint64)
        out["commit_words"] = np.stack([cw & np.uint64(0xFFFFFFFF), cw >> np.uint64(32)], axis=1).astype(np.float64)
        out["commit_bar"] = bar[idx_t].cpu().numpy().view(np.uint32).astype(np.float64)
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in out.items():
        np.save(d / f"{name}.npy", a)


def _max_over_ranks(torch, dist, dev, world, *vals):
    if world == 1:
        return vals if len(vals) > 1 else vals[0]
    t = torch.tensor(list(vals), dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out = [float(x) for x in t]
    return out if len(out) > 1 else out[0]


# =================================================================================================
# GPU arm
# =================================================================================================
def run_ours(args):
    import torch
    import torch.distributed as dist
    from summerset_b200 import sharding, workloads as wl
    from summerset_b200.api import Context, ReedSolomon, SS_RS_OUT_PADDED16
    from summerset_b200._lib import check

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs needs a single process (--gpus 1)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = Context(local)
    rs = ReedSolomon(ctx, D, P)
    rs.set_variant(args.variant)
    n = args.groups
    L, ds, ps = rs.parity_layout(DATA_LEN, n)
    peak, peak_src = measured_peaks()
    env = dict(torch=torch, dist=dist, ctx=ctx, rs=rs, dev=dev, world=world, rank=rank, peak=peak, peak_src=peak_src, args=args)

    # ---- the other configs as the main line (--workload) ----
    if args.workload in ("cfg3b", "cfg4", "cfg5"):
        fn = {"cfg3b": bench_cfg3b, "cfg4": bench_cfg4, "cfg5": bench_cfg5}[args.workload]
        sampler = ClockSampler(local) if rank == 0 else None
        sub = fn(env, args.steps, args.warmup)
        clocks = sampler.stop() if sampler else None
        if rank == 0:
            line = {"metric": sub.pop("metric"), "value": sub.pop("value"), "unit": sub.pop("unit"), "n_gpus": world,
                    "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": sub["ms_per_step"],
                    "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": sub.pop("dtype", "u8"),
                    "data": "synthetic", "config": {"workload": WORKLOAD_TEXT[args.workload], "groups_per_gpu": sub.pop("groups")},
                    "e2e": None, "cpu_baseline": None, "clocks": clocks}
            line.update(sub)
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return

    # ---- synthetic inputs, generated on the device (seeded) ----
    gen = torch.Generator(device=dev); gen.manual_seed(wl.SEED_BASE + 3 + 1000 * rank)
    data = torch.randint(0, 256, (n, DATA_LEN), dtype=torch.uint8, device=dev, generator=gen)
    # ack planes: leader always acks, followers with p = 0.9 (230/256)
    u = torch.randint(0, 256, (R, n, 64), dtype=torch.uint8, device=dev, generator=gen) < 230
    w = torch.tensor([1 << i for i in range(63)] + [-(1 << 63)], dtype=torch.int64, device=dev)
    planes = (u.to(torch.int64) * w).sum(dim=2)
    planes[0] = -1
    del u
    committed = torch.empty(n, dtype=torch.int64, device=dev)
    bar = torch.empty(n, dtype=torch.int32, device=dev)
    parity = None
    rep = None                                       # multi-GPU step state (p2p)
    nccl = None                                      # NCCL all-to-all baseline state
    if world == 1:
        parity = torch.empty((P, n, ds), dtype=torch.uint8, device=dev)
    elif args.exchange in ("p2p", "ce"):
        from summerset_b200.replicate import ReplicatedAcceptStep

        def exchange_handles(obj):
            out = [None] * world
            dist.all_gather_object(out, obj)
            return out
        rep = ReplicatedAcceptStep(ctx, rs, n, DATA_LEN, R, world, rank, exchange_handles, lag=2 if args.exchange == "ce" else args.lag,
                                   mode=args.exchange)
        rep.fill_acks(planes)
        dist.barrier()
    else:
        shards = torch.zeros((D + P, n, ds), dtype=torch.uint8, device=dev)
        nccl = dict(shards=shards, recv=torch.empty((R, n, ds), dtype=torch.uint8, device=dev),
                    ack_recv=planes.clone(), rounds=sharding.exchange_rounds(R, world, rank))
        parity = shards[D:]

    def nccl_exchange():
        sh, recv, ack_recv = nccl["shards"], nccl["recv"], nccl["ack_recv"]
        for rd in nccl["rounds"]:
            ins = [sh[rd["send"][dst]] if rd["send"][dst] >= 0 else sh[0][:0] for dst in range(world)]
            outs = [recv[rd["recv"][src]] if rd["recv"][src] >= 0 else recv[0][:0] for src in range(world)]
            dist.all_to_all(outs, ins)
        for rd in nccl["rounds"]:
            ins = [planes[rd["recv"][src]] if rd["recv"][src] >= 0 else planes[0][:0] for src in range(world)]
            outs = [ack_recv[rd["send"][dst]] if rd["send"][dst] >= 0 else ack_recv[0][:0] for dst in range(world)]
            dist.all_to_all(outs, ins)

    def kernel_only():
        if rep is not None:
            rep.encode_only(data, THRESH_RSPAXOS, committed, bar)
        elif args.workload == "cfg2":
            ctx.tally_planes(planes, THRESH_MULTIPAXOS, True, committed, bar)
        elif args.no_tally:
            check(ctx.lib.ss_rs_encode_uniform_dev(rs.h, data.data_ptr(), DATA_LEN, DATA_LEN, n, parity.data_ptr(), ps, ds, SS_RS_OUT_PADDED16))
        else:
            fl = SS_RS_OUT_PADDED16 | (2 if nccl is not None else 0)
            src = nccl["ack_recv"] if nccl is not None else planes
            check(ctx.lib.ss_accept_step_fused_dev(rs.h, data.data_ptr(), DATA_LEN, DATA_LEN, n, parity.data_ptr(), ps, ds, fl,
                                                   src.data_ptr(), R, THRESH_RSPAXOS, committed.data_ptr(), bar.data_ptr()))

    def step():
        if rep is not None:
            # E_k (tally of the acks of step k - lag, encode, shards stored into the followers' GPUs, shard flags) and
            # A_k (this GPU's followers ack the shards that landed here: ack planes stored into the leaders' GPUs, ack flags)
            rep.step(data, planes, THRESH_RSPAXOS, committed, bar)
            return
        kernel_only()
        if nccl is not None:
            nccl_exchange()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # The clock sampler is started BEFORE the warm-up: forking nvidia-smi takes rank 0's host thread tens of ms, and at N > 1
    # the other ranks' first timed steps would wait that long for rank 0's first launch (profiles/r02_timeline_n8_*_serial*:
    # one 70-100 ms interval at the start of the timed region on every rank but 0 -- the "5 ms/step outside the kernel" of
    # round 1's N = 8 run).
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(max(3, args.warmup)):
        step()
    if rep is not None:
        rep.drain()
    barrier()
    launches0 = ctx.launches + (rep.comm.launches if rep is not None and rep.mode == "ce" else 0)
    tl = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)] if (args.timeline and world > 1) else None
    t_start = torch.cuda.Event(enable_timing=True); t_end = torch.cuda.Event(enable_timing=True)
    t_start.record()
    for i in range(args.steps):
        if tl is not None:
            tl[i].record()
        step()
    if rep is not None:
        rep.drain()                                  # the copy stream's tail belongs to the timed region
    if tl is not None:
        tl[args.steps].record()
    t_end.record()
    barrier()
    total_ms = t_start.elapsed_time(t_end)
    launches = ctx.launches + (rep.comm.launches if rep is not None and rep.mode == "ce" else 0) - launches0
    clocks = sampler.stop() if sampler else None
    status = ctx.device_status()
    assert status == 0, f"device status {status}: a step-flag wait timed out"
    if args.dump_outputs:                            # before the passes below launch the kernels again
        dump_step_outputs(torch, dev, args.dump_outputs, parity if args.workload != "cfg2" else None,
                          committed if (args.workload == "cfg2" or not args.no_tally) else None, bar, n, L)
    # kernel-only duration (CUDA events around the launches), measured in a second pass so the events do not perturb
    # the whole-step timing above
    k_evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for a, b in k_evs:
        a.record(); kernel_only(); b.record()
    torch.cuda.synchronize()
    kernel_ms = sum(a.elapsed_time(b) for a, b in k_evs) / len(k_evs)
    total_ms, kernel_ms = _max_over_ranks(torch, dist, dev, world, total_ms, kernel_ms)
    ms_per_step = total_ms / args.steps
    timed_kernel = rs.last_kernel() if args.workload != "cfg2" else "tally_planes_x2_kernel"     # before the checks launch other kernels
    if tl is not None:
        mine = [tl[i].elapsed_time(tl[i + 1]) for i in range(args.steps)]
        allt = [None] * world
        dist.all_gather_object(allt, mine)
        if rank == 0:
            Path(args.timeline).parent.mkdir(parents=True, exist_ok=True)
            Path(args.timeline).write_text(json.dumps({"n_gpus": world, "lag": args.lag, "steps": args.steps,
                                                       "what": "per rank: CUDA-event time between the starts of consecutive steps (ms), timed region",
                                                       "per_rank_step_ms": allt, "kernel_only_ms_max_over_ranks": kernel_ms,
                                                       "ms_per_step": ms_per_step}))

    # ---- parity check of what was just timed, on EVERY rank (outside the timed region).  (1) every byte of every
    #      plane against a second launch of a DIFFERENT kernel (the flat variant-1 kernel); (2) sampled groups against
    #      the oracle -- used here ONLY as the checker; nothing measured or shipped routes through it. ----
    check_note = None
    if args.workload != "cfg2":
        chk = torch.empty((D + P, n, ds), dtype=torch.uint8, device=dev)
        rs.set_variant(1)
        check(ctx.lib.ss_rs_encode_uniform_dev(rs.h, data.data_ptr(), DATA_LEN, DATA_LEN, n, chk[D].data_ptr(), ps, ds,
                                               SS_RS_OUT_PADDED16 | 2))
        rs.set_variant(args.variant)
        torch.cuda.synchronize()
        if rep is not None:
            got = rep.my_shards()                     # read from the followers' GPUs through the IPC mappings
            ok = all(torch.equal(got[r], chk[r]) for r in range(D + P))
            planes_checked = D + P
        elif nccl is not None:
            ok = torch.equal(nccl["shards"], chk); planes_checked = D + P
        else:
            ok = torch.equal(parity, chk[D:]); planes_checked = P
        assert ok, f"rank {rank}: shard planes differ from the flat-kernel re-encode"
        idx = torch.arange(0, n, max(1, n // 1024), device=dev)
        from oracle import pyoracle as oracle
        want = oracle.rs_encode_uniform(D, P, data[idx].cpu().numpy(), DATA_LEN)
        assert (chk[D:, idx].cpu().numpy() == want).all(), "bench parity check vs oracle failed"
        src = rep.acks_view[rep.k % rep.nbuf] if rep is not None else (nccl["ack_recv"] if nccl is not None else planes)
        if args.no_tally:
            ctx.tally_planes(src, THRESH_RSPAXOS, True, committed, bar)
        # (at N > 1 the last launch -- the kernel-only pass -- tallied the ack buffer the followers' GPUs last wrote)
        cw, bw = oracle.tally_planes(src[:, idx].cpu().numpy().view(np.uint64), THRESH_RSPAXOS)
        assert (committed[idx].cpu().numpy().view(np.uint64) == cw).all(), "bench commit check failed"
        assert (bar[idx].cpu().numpy().view(np.uint32) == bw).all(), "bench commit_bar check failed"
        del chk
        check_note = (f"every byte of {planes_checked} planes x {n} groups == flat-kernel re-encode on every rank; "
                      f"{len(idx)} sampled groups bit-exact vs oracle (parity + commit words + commit_bar)")
    else:
        from oracle import pyoracle as oracle
        idx = torch.arange(0, n, max(1, n // 1024), device=dev)
        cw, bw = oracle.tally_planes(planes[:, idx].cpu().numpy().view(np.uint64), THRESH_MULTIPAXOS)
        assert (committed[idx].cpu().numpy().view(np.uint64) == cw).all(), "bench commit check failed"
        check_note = f"{len(idx)} sampled groups bit-exact vs oracle"
    if world > 1:
        okt = torch.ones(1, device=dev); dist.all_reduce(okt)      # every rank got here => every rank's check passed

    alg_rs = (D + P) * L                       # 6830 B / codeword (SURVEY 8d)
    alg_tally = (R + 1) * 8 + 4                # 48 B planes+commit word, +4 B commit_bar
    if args.workload == "cfg2":
        alg = alg_tally
        value = n * world * 64 / (ms_per_step * 1e-3)
        unit = "slots/s"
    else:
        alg = alg_rs + (0 if args.no_tally else alg_tally)
        value = alg_rs * n * world / (ms_per_step * 1e-3) / 1e9
        unit = "GB/s"
    tkey = (args.workload if R == 5 else f"{args.workload}_r{R}") + ("_5planes" if (world > 1 and args.workload == "cfg3") else "")
    # N > 1: the step also writes the d data-shard planes (every replica's log is a separate buffer), SURVEY 8d "state which"
    alg_kernel = alg + (D * L if (world > 1 and args.workload == "cfg3") else 0)
    roofline = roofline_obj(alg_kernel * n, kernel_ms, peak, peak_src, timed_kernel, tkey)
    if world > 1 and args.workload == "cfg3":
        roofline["note"] = ("kernel = the encode + tally launch alone; in exchange mode ce it writes all five planes to local HBM "
                            "(algorithmic bytes include the three data-shard planes), in mode p2p its stores cross NVLink")
    if world > 1 and args.workload == "cfg3":
        # the same fused kernel WITHOUT the replicate stores (parity to local HBM only): per-GPU compute is flat in N
        lp = torch.empty((P, n, ds), dtype=torch.uint8, device=dev)
        local_ms = _time_steps(torch, lambda: check(ctx.lib.ss_accept_step_fused_dev(
            rs.h, data.data_ptr(), DATA_LEN, DATA_LEN, n, lp.data_ptr(), ps, ds, SS_RS_OUT_PADDED16, planes.data_ptr(), R,
            THRESH_RSPAXOS, committed.data_ptr(), bar.data_ptr())), 10, 3)
        del lp
        roofline["local_only_kernel_ms"] = local_ms
        roofline["local_only_frac"] = alg * n / (local_ms * 1e-3) / 1e9 / peak
        remote = sum(1 for r in range(R) if sharding.replica_rank(rank, r, world) != rank)
        nv_bytes = remote * n * L
        nv_ms = nv_bytes / (NVLINK_REF_GBS * 1e9) * 1e3
        hbm_ms = alg_kernel * n / (peak * 1e9) * 1e3
        roofline["comm"] = {"exchange": ("copy-engine push of staged planes overlapped with the next encode + step flags" if args.exchange == "ce"
                                         else "p2p stores by the encode kernel + step flags") if rep is not None else "nccl all-to-all baseline",
                            "lag": args.lag if rep is not None else None,
                            "remote_planes_per_rank": remote, "nvlink_bytes_per_rank_per_step": nv_bytes,
                            "nvlink_ref_gbs": NVLINK_REF_GBS, "nvlink_bound_ms": nv_ms, "hbm_bound_ms": hbm_ms,
                            "step_ms": ms_per_step, "kernel_ms": kernel_ms,
                            "nvlink_gbs_per_step": nv_bytes / (ms_per_step * 1e-3) / 1e9,
                            "nvlink_gbs_in_kernel": nv_bytes / (kernel_ms * 1e-3) / 1e9 if args.exchange == "p2p" else None,
                            "frac_of_slower_bound": max(nv_ms, hbm_ms) / ms_per_step,
                            "note": "target time = slower of HBM bytes / measured copy bandwidth and NVLink bytes / 770 GB/s "
                                    "(measured peer-copy reference, B200_PROFILING.md)"}
    if rank == 0:
        here = copy_bandwidth_here(torch, dev)
        if here:
            roofline["copy_gbs_this_box"] = here
            roofline["frac_of_copy_this_box"] = roofline["achieved"] / here

    # ---- end to end through the host-buffer C-ABI call ----
    e2e = None
    if not args.no_e2e:
        e2e = bench_e2e(env, data, n)

    # free the cfg3 state before the sub-benches (cfg4 needs ~70 GB)
    if rep is not None:
        if world > 1:
            dist.barrier()
        rep.close()
    del data, parity, nccl
    torch.cuda.empty_cache()

    extra = {}
    if args.workload == "cfg3" and not args.no_sub and R == 5:
        sub_steps = 20
        if world == 1:
            extra["cfg2"] = bench_cfg2(env, n)
            extra["cfg3b"] = bench_cfg3b(env, sub_steps, 3)
            torch.cuda.empty_cache()
        extra["cfg4"] = bench_cfg4(env, 10 if world == 1 else 8, 3)
        torch.cuda.empty_cache()
        extra["cfg5"] = bench_cfg5(env, sub_steps, 3)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        # the CPU arm in its own process (its OpenMP binding must not touch this one): the reference line's cpu_baseline
        try:
            out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "5", "--warmup", "1",
                                  "--workload", args.workload, "--groups", str(n), "--replicas", str(R)],
                                 capture_output=True, text=True, timeout=600)
            cpu = json.loads(out.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as ex:                         # reported, never silently dropped
            cpu = {"value": None, "unit": unit, "cores": 0, "kind": "port", "sample": f"CPU arm failed: {ex!r}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": config_dict(args, world),
            "slots_committed_per_s": n * world * 64 / (ms_per_step * 1e-3),
            "payload_GBps": DATA_LEN * n * world / (ms_per_step * 1e-3) / 1e9,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "parity_check": check_note,
        }
        if world > 1 and args.workload == "cfg3":
            line["scaling_note"] = ("N=1 simulates all 5 replicas of a group on one GPU (no exchange: the shard planes are the "
                                    "follower logs). At N>1 replica r of a group led from rank h lives on rank (h+r)%N and the encode "
                                    "kernel stores its shard there over NVLink, so the step becomes NVLink-bound (roofline.comm); the "
                                    "same kernel without the remote stores takes roofline.local_only_kernel_ms on every N.")
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# =================================================================================================
# sub-benches (each returns a dict; also usable as the main line through --workload)
# =================================================================================================
def bench_cfg2(env, n):
    torch, ctx, dev, peak = env["torch"], env["ctx"], env["dev"], env["peak"]
    sets = 4
    gen = torch.Generator(device=dev); gen.manual_seed(1234)
    planes = torch.randint(-(1 << 62), 1 << 62, (sets, R, n), dtype=torch.int64, device=dev, generator=gen)
    planes[:, 0] = -1
    committed = torch.empty((sets, n), dtype=torch.int64, device=dev)
    bar = torch.empty((sets, n), dtype=torch.int32, device=dev)
    for i in range(8):
        ctx.tally_planes(planes[i % sets], THRESH_MULTIPAXOS, True, committed[i % sets], bar[i % sets])
    torch.cuda.synchronize()
    iters = 40
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        ctx.tally_planes(planes[i % sets], THRESH_MULTIPAXOS, True, committed[i % sets], bar[i % sets])
    b.record()
    torch.cuda.synchronize()
    ms_plain = a.elapsed_time(b) / iters
    # The launch is ~10 us of work: back-to-back launches from the host leave a gap of a few us between kernels.  A
    # CUDA graph of the four rotated launches removes most of it (the engine's tick would be captured the same way).
    ms = ms_plain
    graphed = False
    try:
        from summerset_b200.api import Context
        side = torch.cuda.Stream(device=dev)
        with torch.cuda.stream(side):
            gctx = Context(dev.index)                     # a context on the capturing stream
            for i in range(sets):
                gctx.tally_planes(planes[i], THRESH_MULTIPAXOS, True, committed[i], bar[i])
            side.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side, capture_error_mode="thread_local"):
                for i in range(sets):
                    gctx.tally_planes(planes[i], THRESH_MULTIPAXOS, True, committed[i], bar[i])
            for _ in range(3):
                graph.replay()
            side.synchronize()
            a.record(side)
            for _ in range(iters // sets):
                graph.replay()
            b.record(side)
            side.synchronize()
            ms = a.elapsed_time(b) / iters
            graphed = True
            gctx.close()
    except Exception as ex:                               # capture unsupported: keep the plain figure, and say so
        graph_note = f"CUDA graph capture failed ({ex!r}); plain launches"
    else:
        graph_note = "40 launches as 10 replays of a CUDA graph of the 4 rotated launches"
    alg = ((R + 1) * 8 + 4) * n
    return {"workload": WORKLOAD_TEXT["cfg2"] + ", 4 rotated plane sets (208 MB > L2)",
            "slots_committed_per_s": n * 64 / (ms * 1e-3), "ms_per_step": ms, "ms_per_step_plain_launches": ms_plain,
            "cuda_graph": graphed, "timing": graph_note,
            "roofline": roofline_obj(alg, ms, peak, env["peak_src"], "tally_planes_x2_kernel", "cfg2",
                                     note="52 B/group; 8.4 us of traffic per launch at the copy bandwidth, 10.7 us kernel under ncu; the rest is launch gap")}


def bench_e2e(env, data_dev, n):
    """Same step through the host-buffer C-ABI entry point ss_accept_step_fused: pinned host payloads + ack planes in,
    parity + commit words + commit_bar out; H2D + ONE fused kernel per chunk + D2H inside the timed region.  The
    process is bound to the GPU's NUMA node while the pinned buffers are allocated and the calls are made."""
    torch, dist, ctx, rs, dev, world, rank, args = (env[k] for k in ("torch", "dist", "ctx", "rs", "dev", "world", "rank", "args"))
    L, ds, ps = rs.parity_layout(DATA_LEN, n)
    steps = max(3, min(args.steps, 10))
    pin = NumaPin(torch, dev.index)
    with pin:
        hplanes = torch.empty((R, n), dtype=torch.int64, pin_memory=True)
        hplanes.random_(-(1 << 62), 1 << 62)
        hplanes[0] = -1
        pn = hplanes.numpy().view(np.uint64)
        hcm = torch.empty(n, dtype=torch.int64, pin_memory=True)
        hbar = torch.empty(n, dtype=torch.int32, pin_memory=True)
        if args.workload == "cfg2":
            ctx.tally_planes_host(pn, THRESH_MULTIPAXOS)
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                ctx.tally_planes_host(pn, THRESH_MULTIPAXOS)
            dt = (time.perf_counter() - t0) / steps
            dt = _max_over_ranks(torch, dist, dev, world, dt)
            return {"value": n * world * 64 / dt, "unit": "slots/s", "h2d_bytes_per_step": R * n * 8,
                    "d2h_bytes_per_step": n * 12, "steps": steps, "ms_per_step": dt * 1e3}
        hdata = torch.empty((n, DATA_LEN), dtype=torch.uint8, pin_memory=True)
        hdata.copy_(data_dev)                           # the device-generated synthetic payloads, now in pinned host memory
        torch.cuda.synchronize()
        hv = hdata.numpy()
        hpar = torch.empty((P, n, ds), dtype=torch.uint8, pin_memory=True)
        cm = hcm.numpy().view(np.uint64); bn = hbar.numpy().view(np.uint32)

        def step():
            rs.accept_step_fused_host(hv, DATA_LEN, hpar.numpy(), pn, THRESH_RSPAXOS, cm, bn)

        step()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = (time.perf_counter() - t0) / steps
    dt = _max_over_ranks(torch, dist, dev, world, dt)
    # check the e2e result too (oracle as the checker)
    from oracle import pyoracle as oracle
    idx = np.arange(0, n, max(1, n // 256))
    want = oracle.rs_encode_uniform(D, P, hv[idx], DATA_LEN)
    assert (hpar.numpy()[:, idx] == want).all(), "e2e parity check failed"
    cw, bw = oracle.tally_planes(np.ascontiguousarray(pn[:, idx]), THRESH_RSPAXOS)
    assert (cm[idx] == cw).all() and (bn[idx] == bw).all(), "e2e commit check failed"
    return {"value": (D + P) * L * n * world / dt / 1e9, "unit": "GB/s",
            "h2d_bytes_per_step": n * DATA_LEN + R * n * 8, "d2h_bytes_per_step": P * n * ds + n * 12,
            "steps": steps, "ms_per_step": dt * 1e3, "slots_committed_per_s": n * world * 64 / dt,
            "per_gpu_value": (D + P) * L * n / dt / 1e9, "numa_node": pin.node, "numa_pinned": bool(pin.cpus),
            "call": "ss_accept_step_fused (payload + ack planes H2D, fused encode+tally kernel per 16 MiB chunk, parity + commit words + commit_bar D2H)",
            "timing": "host wall clock around the blocking C-ABI call (returns when results are in host memory); max over ranks"}


def bench_cfg5(env, steps, warmup):
    torch, dist, ctx, dev, world, rank, peak = (env[k] for k in ("torch", "dist", "ctx", "dev", "world", "rank", "peak"))
    from summerset_b200 import workloads as wl
    G = 1 << 22
    w = wl.cfg5_raft(1 << 16, 7, 64, seed_extra=rank)
    rep = G // (1 << 16)
    t = lambda a, r: torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).to(dev).repeat(*r)
    match = t(w["match"], (1, rep)); lc = t(w["last_commit"], (rep,)); le = t(w["log_end"], (rep,))
    ct = t(w["curr_term"], (rep,)); terms = t(w["terms"], (rep, 1))
    out = torch.empty(G, dtype=torch.int32, device=dev)
    ovf = torch.zeros(1, dtype=torch.int32, device=dev)
    l0 = ctx.launches
    ms = _time_steps(torch, lambda: ctx.raft_commit_scan(match, lc, le, ct, terms, 4, out, ovf), steps, warmup)
    launches = (ctx.launches - l0) * steps // (steps + max(3, warmup))
    ms = _max_over_ranks(torch, dist, dev, world, ms)
    from oracle import pyoracle as oracle
    want = oracle.raft_scan_batch(w["match"], w["last_commit"], w["log_end"], w["curr_term"], w["terms"], 4)
    assert (out[:1 << 16].cpu().numpy().view(np.uint32) == want).all() and int(ovf) == 0, "cfg5 check failed"
    alg = 296 * G
    return {"metric": "Raft groups scanned/s (7 replicas, 64-slot window)", "value": G * world / (ms * 1e-3), "unit": "groups/s",
            "dtype": "u32", "groups": G, "workload": WORKLOAD_TEXT["cfg5"], "ms_per_step": ms, "n_gpus": world,
            "parity_check": "first 2^16 groups (the tile the batch repeats) bit-exact vs oracle",
            "roofline": roofline_obj(alg, ms, peak, env["peak_src"], "raft_scan_kernel", "cfg5",
                                     note="charged 296 B/group (SURVEY 8d); the probe path reads fewer term words"),
            "gpu_launches": int(launches)}


def bench_cfg3b(env, steps, warmup):
    """cfg 3b: batched reconstruct_data of 2^20 RS(3,2) codewords x 4 KB under the seeded erasure mix."""
    torch, ctx, rs, dev, world, rank, peak, args = (env[k] for k in ("torch", "ctx", "rs", "dev", "world", "rank", "peak", "args"))
    from summerset_b200 import workloads as wl
    n = args.groups
    L, ds, ps = rs.parity_layout(DATA_LEN, n)
    gen = torch.Generator(device=dev); gen.manual_seed(wl.SEED_BASE + 3 + rank)
    data = torch.randint(0, 256, (n, DATA_LEN), dtype=torch.uint8, device=dev, generator=gen)
    sh = torch.zeros((D + P, n, ds), dtype=torch.uint8, device=dev)
    padded = torch.zeros((n, D * L), dtype=torch.uint8, device=dev)
    padded[:, :DATA_LEN] = data
    for i in range(D):
        sh[i, :, :L] = padded[:, i * L:(i + 1) * L]
    del padded
    rs.encode_uniform(data, DATA_LEN, parity=sh[D:])
    del data
    keep = sh[:D].clone()
    present = wl.erasure_patterns(n, D, P, seed_extra=rank)
    pm = torch.from_numpy(present.astype(np.int32)).to(dev)
    for j in range(D + P):
        sh[j][((pm >> j) & 1) == 0] = 0x5A
    l0 = ctx.launches
    ms = _time_steps(torch, lambda: rs.reconstruct_uniform(sh, DATA_LEN, pm, True), steps, warmup)
    launches = (ctx.launches - l0) * steps // (steps + max(3, warmup))
    ok = all(torch.equal(sh[i], keep[i]) for i in range(D))
    assert ok, "cfg3b round trip failed"
    miss_data = sum(((present >> i) & 1) == 0 for i in range(D)).astype(np.int64)
    alg = int(((miss_data > 0) * D * L + miss_data * L).sum()) + n * 20
    kernel = rs.last_kernel()
    del sh, keep
    return {"metric": "RS reconstruct GB/s (reconstruct_data, RS(3,2), 4 KB payloads, cfg-3b erasure mix)",
            "value": alg / (ms * 1e-3) / 1e9, "unit": "GB/s", "groups": n, "workload": WORKLOAD_TEXT["cfg3b"], "ms_per_step": ms,
            "codewords_per_s": n / (ms * 1e-3), "roundtrip_bit_exact": bool(ok),
            "parity_check": "every regenerated data shard of every codeword == the original (encode -> erase -> reconstruct)",
            "roofline": roofline_obj(alg, ms, peak, env["peak_src"], kernel, "cfg3b"), "gpu_launches": int(launches)}


def bench_cfg4(env, steps, warmup):
    """cfg 4: Crossword n=5,d=3,T=5,f=2: ragged RS(3,2) encode of mixed 256 B..64 KB payloads, shards distributed by
    the balanced round-robin assignment into the five replica logs (local or peer GPUs), + coverage tally."""
    torch, dist, ctx, rs, dev, world, rank, peak, args = (env[k] for k in ("torch", "dist", "ctx", "rs", "dev", "world", "rank", "peak", "args"))
    from oracle import pyoracle as oracle
    from summerset_b200 import sharding, workloads as wl
    from summerset_b200.api import crossword_brr_assignment, cw_slot_pitch
    n = args.groups
    lens, spr = wl.cfg4_lengths(n, seed_extra=0)      # same sizes on every rank (payload bytes differ by rank)
    lay = wl.ragged_layout(lens, D)
    gen = torch.Generator(device=dev); gen.manual_seed(wl.SEED_BASE + 4 + rank)
    arena = torch.randint(0, 256, (lay["data_bytes"] + 256,), dtype=torch.uint8, device=dev, generator=gen)
    parity = torch.empty((P, lay["plane_bytes"]), dtype=torch.uint8, device=dev)
    doff = torch.from_numpy(lay["data_off"].astype(np.int64)).to(dev)
    poff = torch.from_numpy(lay["par_off"].astype(np.int64)).to(dev)
    dlen = torch.from_numpy(lens.astype(np.int32)).to(dev)
    masks = torch.randint(0, 32, (n,), dtype=torch.uint8, device=dev, generator=gen) | 1     # leader always acks
    pidx = torch.from_numpy((spr - 1).astype(np.uint8)).to(dev)
    policies = [crossword_brr_assignment(5, 5, s) for s in (1, 2, 3)]
    # replica logs for the distribute step: replica r of my groups lives on rank (rank + r) % world
    Lp = cw_slot_pitch(lay["L"].astype(np.int64))
    slot_bytes = spr.astype(np.int64) * Lp
    rep_off_np = np.concatenate([[0], np.cumsum(slot_bytes)[:-1]]).astype(np.int64)
    region = int(slot_bytes.sum() + 255) // 256 * 256
    log = ctx.dev_alloc(5 * region)
    peer_log = {rank: log}
    tiny = None
    if world > 1:
        handles = [None] * world
        dist.all_gather_object(handles, ctx.ipc_export(log))
        for q in range(world):
            if q != rank:
                peer_log[q] = ctx.ipc_open(handles[q], 5 * region)
        tiny = torch.zeros(1, dtype=torch.int32, device=dev)
    rep_ptrs = [peer_log[sharding.replica_rank(rank, r, world)].ptr + r * region for r in range(5)]
    rep_off = torch.from_numpy(rep_off_np).to(dev)
    spr_t = torch.from_numpy(spr).to(dev)

    def step():
        # lens were drawn with the same seed on every rank, so all regions have the same size
        rs.crossword_distribute(arena, doff, dlen, spr_t, rep_off, rep_ptrs)
        out = ctx.tally_crossword(masks, pidx, policies, 5, 3, 3, 2, True)
        if world > 1:
            dist.all_reduce(tiny)
        return out

    l0 = ctx.launches
    ms = _time_steps(torch, step, steps, warmup)
    launches = (ctx.launches - l0) * steps // (steps + max(3, warmup))
    dist_kernel = rs.last_kernel()
    ms_dist = _time_steps(torch, lambda: rs.crossword_distribute(arena, doff, dlen, spr_t, rep_off, rep_ptrs), steps, 1) if world == 1 else None
    ms_enc = _time_steps(torch, lambda: rs.encode_batch(arena, doff, dlen, parity, lay["plane_bytes"], poff), steps, 1)
    enc_kernel = rs.last_kernel()
    ms, ms_enc = _max_over_ranks(torch, dist, dev, world, ms, ms_enc)
    # the follower view: replica 1 of my groups (wherever it lives) holds shard (1 + k) % 5 in slot k
    chk = peer_log[sharding.replica_rank(rank, 1, world)].tensor()[region:2 * region]
    idx = np.arange(0, n, max(1, n // 64))
    sub_len = lens[idx]; sub_lay = wl.ragged_layout(sub_len, D)
    sub = np.zeros(sub_lay["data_bytes"] + 64, dtype=np.uint8)
    for j, g in enumerate(idx):
        o = int(lay["data_off"][g]); so = int(sub_lay["data_off"][j]); ln = int(lens[g])
        sub[so:so + ln] = arena[o:o + ln].cpu().numpy()
    want = np.zeros((P, sub_lay["plane_bytes"]), dtype=np.uint8)
    oracle.rs_encode_batch(D, P, sub, sub_lay["data_off"], sub_len, want.reshape(-1), sub_lay["plane_bytes"], sub_lay["par_off"])
    for j, g in enumerate(idx):
        Lg = int(lay["L"][g]); o = int(lay["par_off"][g]); so = int(sub_lay["par_off"][j])
        got = parity[:, o:o + Lg].cpu().numpy()
        assert (got == want[:, so:so + Lg]).all(), "cfg4 parity check failed"
        if spr[g] == 3:     # replica 1, slot 2 = shard 3 = parity 0
            o2 = int(rep_off_np[g]) + 2 * int(Lp[g])
            assert (chk[o2:o2 + Lg].cpu().numpy() == want[0, so:so + Lg]).all(), "cfg4 distribute check failed"
    note = f"{len(idx)} sampled codewords bit-exact vs oracle (parity planes and replica-1 log)"
    alg = int((lay["L"].astype(np.int64) * (D + P)).sum()) + n * 22
    alg_dist = int((lay["L"].astype(np.int64) * (D + 5 * spr.astype(np.int64))).sum()) + n * 31
    remote = sum(1 for r in range(5) if sharding.replica_rank(rank, r, world) != rank)
    nv_bytes = int((lay["L"].astype(np.int64) * spr.astype(np.int64)).sum()) * remote
    nv_ms = nv_bytes / (NVLINK_REF_GBS * 1e9) * 1e3
    hbm_ms = alg_dist / (peak * 1e9) * 1e3
    res = {"metric": "RS shard GB/s, Crossword ragged encode + distribute-by-assignment + coverage tally",
           "value": alg * world / (ms * 1e-3) / 1e9, "unit": "GB/s", "groups": n, "workload": WORKLOAD_TEXT["cfg4"], "n_gpus": world,
           "ms_per_step": ms, "payload_bytes": int(lens.astype(np.int64).sum()),
           "distribute": {"kernel": dist_kernel, "step_ms": ms, "kernel_ms": ms_dist, "hbm_bytes_per_rank": alg_dist,
                          "hbm_GBps_per_rank": alg_dist / (ms * 1e-3) / 1e9,
                          "nvlink_bytes_per_rank": nv_bytes, "nvlink_bound_ms": nv_ms, "hbm_bound_ms": hbm_ms,
                          "frac_of_slower_bound": max(nv_ms, hbm_ms) / ms,
                          "roofline": roofline_obj(alg_dist, ms_dist, peak, env["peak_src"], dist_kernel, "cfg4_distribute") if ms_dist else None},
           "slots_committed_per_s": n * world / (ms * 1e-3), "encode_only_ms": ms_enc, "parity_check": note,
           "roofline": roofline_obj(alg, ms_enc, peak, env["peak_src"], enc_kernel, "cfg4"), "gpu_launches": int(launches)}
    if world > 1:
        dist.barrier()
        for q in peer_log:
            if q != rank:
                peer_log[q].free()
        dist.barrier()
    log.free()
    del arena, parity
    return res


def main():
    global D, P, R, THRESH_RSPAXOS, THRESH_MULTIPAXOS
    args = parse_args()
    # The contract is ONE JSON line on stdout.  Native libraries print there too (NCCL writes "NCCL version ..." to fd 1
    # when the first communicator comes up), so fd 1 is pointed at stderr for the whole run and Python's sys.stdout
    # keeps a private duplicate of the real stdout for the result line.
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    if args.replicas != 5:      # scripts/local_cluster.py:41-50 defaults: fault_tolerance = (n//2)//2
        R = args.replicas
        D = R // 2 + 1
        P = R - D
        THRESH_MULTIPAXOS = D
        THRESH_RSPAXOS = D + (R // 2) // 2
    if args.rs:
        D, P = (int(x) for x in args.rs.split(","))
        R = D + P
        THRESH_MULTIPAXOS = R // 2 + 1
        THRESH_RSPAXOS = min(R, R // 2 + 1 + (R // 2) // 2)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
