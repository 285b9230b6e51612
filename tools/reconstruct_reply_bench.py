"""ss_reconstruct_reply_dev on one GPU: a follower's window of 2^14 groups x 64 instances of RS(3,2) with 4 KB request
batches receives its Reconstruct replies.

Workload: the follower (replica 1) holds its own shard of every instance; two other replicas each send one shard per
instance (a random pair of {0, 2, 3, 4}), replies grouped per sending peer as ss_reconstruct_serve_dev writes them, plus
5 % retransmitted duplicates at the end.  Every instance is committed and every bar starts at 0, so the walk passes all
64 instances of every group and decodes the 5 in 6 that lack a data shard.  The reply bytes (~2.9 GB) are far above the
126 MB L2.

Timing: CUDA events around each call (warm-up first, >= 100 timed calls); present and exec_bar are restored between
calls outside the events.  The three kernels of one call (absorb, walk, decode) are split by torch.profiler in a run of
its own.  Bytes are algorithmic, computed from the shapes below; fractions are of the 6489.3 GB/s copy bandwidth
DESIGN.md uses, and a device-to-device copy of the reply buffer is timed in the same run for comparison.

Usage: python tools/reconstruct_reply_bench.py [--groups N] [--iters K] [--warmup W] [--out file.json]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

PEAK_GBS = 6489.3
KERNELS = {"absorb": "reconstruct_absorb_kernel", "walk": "reconstruct_walk_kernel", "decode": "rs32_reconstruct_row_kernel"}


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                          # the figures below are meaningless without the card beside them
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})", "max_sm_clock": "unavailable"}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--groups", type=int, default=1 << 14)
    ap.add_argument("--window", type=int, default=64)
    ap.add_argument("--data-len", type=int, default=4096)
    ap.add_argument("--dup", type=float, default=0.05)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", type=str, default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a GPU: nothing here is measured on the CPU")

    from summerset_b200 import _lib
    from summerset_b200.api import Context, ReedSolomon, _ptr

    torch.cuda.set_device(0)
    dev = "cuda:0"
    ctx = Context(0)
    d, p, me = 3, 2, 1
    T = d + p
    rs = ReedSolomon(ctx, d, p)
    G, W, data_len = a.groups, a.window, a.data_len
    n = G * W
    L = (data_len + d - 1) // d
    slot = (L + 15) // 16 * 16
    gen = torch.Generator(device=dev)
    gen.manual_seed(1)

    # the codewords: payloads encoded into T planes (data shards emitted too); the follower's shard store IS these planes,
    # so absorbed and regenerated slots are rewritten with the bytes already there and the store stays valid call to call
    stride = (data_len + 15) // 16 * 16
    payload = torch.randint(0, 256, (n, stride), dtype=torch.uint8, device=dev, generator=gen)
    planes = torch.empty((T, n, slot), dtype=torch.uint8, device=dev)
    _lib.check(rs.lib.ss_rs_encode_uniform_dev(rs.h, _ptr(payload), stride, data_len, n, planes[d].data_ptr(), n * slot,
                                               slot, _lib.SS_RS_OUT_PADDED16 | 2))                   # | SS_RS_EMIT_DATA
    del payload

    # two single-shard replies per instance from a random pair of the other replicas, grouped per sending peer
    others = torch.tensor([j for j in range(T) if j != me], device=dev)
    pick = others[torch.rand((n, T - 1), device=dev, generator=gen).argsort(dim=1)[:, :2]]         # [n, 2]
    rows_all = torch.arange(n, device=dev)
    inst, shard = [], []
    for q in others.tolist():
        sel = rows_all[(pick == q).any(dim=1)]
        inst.append(sel)
        shard.append(torch.full_like(sel, q))
    inst, shard = torch.cat(inst), torch.cat(shard)
    n_dup = int(round(a.dup * inst.numel()))
    dup = torch.randint(0, inst.numel(), (n_dup,), device=dev, generator=gen)
    inst, shard = torch.cat([inst, inst[dup]]), torch.cat([shard, shard[dup]])
    R = inst.numel()
    reply_buf = planes.view(T * n, slot)[shard * n + inst].reshape(-1)
    reply_off = torch.arange(R, dtype=torch.int64, device=dev) * slot
    reply_mask = (1 << shard).to(torch.int32)
    reply_inst = inst.to(torch.int32)
    reply_ballot = torch.ones(R, dtype=torch.int64, device=dev)
    inst_status = torch.full((n,), 3, dtype=torch.uint8, device=dev)                 # Committed
    inst_bal = torch.ones(n, dtype=torch.int64, device=dev)
    present0 = torch.full((n,), 1 << me, dtype=torch.int32, device=dev)
    bar0 = torch.zeros(G, dtype=torch.int32, device=dev)
    present, bar = present0.clone(), bar0.clone()

    def call():
        return rs.reconstruct_reply(planes, data_len, W, inst_status, inst_bal, present, bar, reply_buf, reply_off, reply_mask,
                                    reply_inst, reply_ballot)

    # one checked call first: the walk passes everything, present ends full of data bits, nothing is taken twice
    submit, taken = call()
    torch.cuda.synchronize()
    assert int(bar.min()) == W and bool((submit == (-1 if W == 64 else (1 << W) - 1)).all())
    assert int(((present & 7) != 7).sum()) == 0
    assert int(taken.ne(0).sum()) == 2 * n

    # algorithmic bytes from the shapes
    dmask = (1 << d) - 1
    got = (1 << me) | (1 << pick[:, 0]) | (1 << pick[:, 1])
    need = (got & dmask) != dmask
    n_dec = int(need.sum())
    missing = int((d - ((got & dmask).view(-1, 1) >> torch.arange(d, device=dev) & 1).sum(dim=1))[need].sum())
    bytes_absorb = R * slot + 2 * n * slot + R * (8 + 4 + 4 + 8 + 4) + R * (1 + 8 + 8)
    bytes_walk = n * (4 + 1 + 4) + n_dec * 4 + G * (4 + 4 + 8)
    bytes_decode = n * (4 + 4) + n_dec * d * slot + missing * slot
    total_bytes = bytes_absorb + bytes_walk + bytes_decode

    # CUDA events around each call; state restored outside them
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(a.iters)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(a.iters)]
    for i in range(a.warmup + a.iters):
        present.copy_(present0)
        bar.copy_(bar0)
        if i >= a.warmup:
            starts[i - a.warmup].record()
        call()
        if i >= a.warmup:
            ends[i - a.warmup].record()
    torch.cuda.synchronize()
    ms = np.array([s.elapsed_time(e) for s, e in zip(starts, ends)])

    # the same-size device-to-device copy, for comparison
    dst = torch.empty_like(reply_buf)
    for _ in range(3):
        dst.copy_(reply_buf)
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(20):
        dst.copy_(reply_buf)
    c1.record()
    torch.cuda.synchronize()
    copy_gbs = 2 * reply_buf.numel() * 20 / (c0.elapsed_time(c1) * 1e-3) / 1e9
    del dst

    # per-kernel split in a profiler run of its own
    from torch.profiler import ProfilerActivity, profile
    n_prof = 20
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_prof):
            present.copy_(present0)
            bar.copy_(bar0)
            call()
        torch.cuda.synchronize()
    per_kernel = {}
    for e in prof.key_averages():
        for k, name in KERNELS.items():
            if name in e.key:
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                per_kernel[k] = per_kernel.get(k, 0.0) + t / 1e3 / n_prof       # ms per call
    kbytes = {"absorb": bytes_absorb, "walk": bytes_walk, "decode": bytes_decode}

    res = {
        "what": "ss_reconstruct_reply_dev, RS(3,2), follower holds 1 shard, 2 single-shard replies per instance + dups",
        **card(),
        "groups": G, "window": W, "instances": n, "data_len": data_len, "slot_bytes": slot,
        "replies": R, "duplicates": n_dup, "reply_bytes": R * slot, "decoded_rows": n_dec, "regenerated_shards": missing,
        "timed_calls": a.iters, "warmup_calls": a.warmup,
        "call_ms_median": float(np.median(ms)), "call_ms_min": float(ms.min()), "call_ms_max": float(ms.max()),
        "algorithmic_bytes": {**kbytes, "total": total_bytes},
        "call_gbs": total_bytes / (np.median(ms) * 1e-3) / 1e9,
        "call_fraction_of_6489": total_bytes / (np.median(ms) * 1e-3) / 1e9 / PEAK_GBS,
        "kernel_ms_profiler": per_kernel,
        "kernel_fraction_of_6489": {k: kbytes[k] / (per_kernel[k] * 1e-3) / 1e9 / PEAK_GBS for k in per_kernel if per_kernel[k] > 0},
        "d2d_copy_gbs_this_box": copy_gbs,
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")
    rs.close()
    ctx.close()


if __name__ == "__main__":
    main()
