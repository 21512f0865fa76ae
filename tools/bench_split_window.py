#!/usr/bin/env python
"""Chunk-parallel inflate of streams whose pieces share history (ZLB_INFLATE_SPLIT, window mode), device resident.

    python tools/bench_split_window.py [--seconds S] [--only NAME,...]  -> one JSON line on stdout

Cases (all inputs made from seeds; every output is compared with the input):
  primed_mixed_256m   synth.mixed(256 MiB, 1), deflated on the GPU in ZLB_MODE_PRIMED (32 KiB chunks, each searching the
                      32 KiB in front of it)
  primed_text_256m    synth.text(256 MiB, 2), the same
  primed_byte_256m    256 MiB of one repeated byte, the same: nearly every byte of a piece comes from the one before
                      (256 MiB, not 64: the split looks at items of at least 256 KiB of compressed input, and 64 MiB
                      of one byte compresses to ~140 KiB, which one warp decodes)
  zlib_sync_64m       synth.mixed(64 MiB, 3) through CPython zlib level 6 with a Z_SYNC_FLUSH every 64 KiB
  compat_mixed_256m   the data of primed_mixed_256m in ZLB_MODE_COMPAT: independent pieces, the split route without
                      window mode (the comparison the window cases are measured against)
  one_warp_primed_16m synth.mixed(16 MiB, 1) in ZLB_MODE_PRIMED without ZLB_INFLATE_SPLIT: what primed streams got
                      before window mode
Timing: one warm-up call, then as many calls as fit in --seconds (at least two) on a host clock; zlb_inflate_batch
ends in a stream synchronise. Outputs of 256 MiB do not fit the 126 MB L2. The per-kernel split comes from one more
call with the profile slots on (kernel milliseconds bracketed by CUDA events), not from the timed calls.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

import zlibts_b200 as z
from zlibts_b200 import synth

MIB = 1 << 20


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = "not read: %s" % e
    return info


def deflate_on_gpu(eng, d_in, mode):
    cap = z.deflate_bound(d_in.numel(), 0, z.DYNAMIC, mode)
    items = z.make_items(1)
    items["in_len"], items["out_cap"] = d_in.numel(), cap
    d_z = torch.empty(cap, dtype=torch.uint8, device="cuda")
    r = eng.deflate_batch(d_in, d_z, items, mode=mode)
    assert int(r["status"][0]) == 0
    return d_z[:int(r["out_len"][0])].clone()


def measure(eng, name, d_in, d_z, flags, seconds):
    n = d_in.numel()
    items = z.make_items(1)
    items["in_len"], items["out_cap"] = d_z.numel(), n
    d_out = torch.empty(n, dtype=torch.uint8, device="cuda")
    r = eng.inflate_batch(d_z, d_out, items, flags)  # warm-up (scratch allocations)
    assert int(r["status"][0]) == 0 and int(r["out_len"][0]) == n, (name, r)
    assert torch.equal(d_out, d_in), name
    d_out.fill_(0)
    reps, t0 = 0, time.perf_counter()
    while True:
        r = eng.inflate_batch(d_z, d_out, items, flags)
        reps += 1
        el = time.perf_counter() - t0
        if reps >= 2 and el >= seconds:
            break
    assert int(r["status"][0]) == 0 and torch.equal(d_out, d_in), name
    eng.profile_enable(True)
    eng.profile_reset()
    eng.inflate_batch(d_z, d_out, items, flags)
    prof = eng.profile_read()
    eng.profile_enable(False)
    kernels = {k: {"ms": round(v["ms"], 3), "launches": v["launches"]} for k, v in prof.items() if v["launches"]}
    ms = el * 1e3 / reps
    return {"case": name, "out_bytes": n, "in_bytes": d_z.numel(), "ms_per_call": round(ms, 3),
            "GBps": round(n / (ms * 1e-3) / 1e9, 3), "calls": reps, "kernels_one_call": kernels,
            "output_equals_input": True}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0, help="least wall time of the timed calls per case")
    ap.add_argument("--only", default="", help="comma-separated case names (default: all)")
    args = ap.parse_args()
    only = set(filter(None, args.only.split(",")))
    eng = z.Engine(0)
    split = z.INFLATE_SPLIT
    out = {"bench": "split_window", **gpu_info(), "cases": []}

    def want(name):
        return not only or name in only

    mixed = torch.from_numpy(synth.mixed(256 * MIB, 1)).cuda()
    if want("primed_mixed_256m"):
        out["cases"].append(measure(eng, "primed_mixed_256m", mixed, deflate_on_gpu(eng, mixed, z.MODE_PRIMED), split,
                                    args.seconds))
    if want("compat_mixed_256m"):
        out["cases"].append(measure(eng, "compat_mixed_256m", mixed, deflate_on_gpu(eng, mixed, z.MODE_COMPAT), split,
                                    args.seconds))
    if want("one_warp_primed_16m"):
        m16 = mixed[:16 * MIB].clone()
        out["cases"].append(measure(eng, "one_warp_primed_16m", m16, deflate_on_gpu(eng, m16, z.MODE_PRIMED), 0, 0.0))
        del m16
    del mixed
    if want("primed_text_256m"):
        text = torch.from_numpy(synth.text(256 * MIB, 2)).cuda()
        out["cases"].append(measure(eng, "primed_text_256m", text, deflate_on_gpu(eng, text, z.MODE_PRIMED), split,
                                    args.seconds))
        del text
    if want("primed_byte_256m"):
        byte = torch.full((256 * MIB,), 0x61, dtype=torch.uint8, device="cuda")
        out["cases"].append(measure(eng, "primed_byte_256m", byte, deflate_on_gpu(eng, byte, z.MODE_PRIMED), split,
                                    args.seconds))
        del byte
    if want("zlib_sync_64m"):
        h = synth.mixed(64 * MIB, 3).tobytes()
        co = zlib.compressobj(6, zlib.DEFLATED, -15)
        s = b"".join(co.compress(h[k:k + 65536]) + co.flush(zlib.Z_SYNC_FLUSH) for k in range(0, len(h), 65536))
        s += co.flush()
        d_s = torch.from_numpy(np.frombuffer(s, dtype=np.uint8).copy()).cuda()
        out["cases"].append(measure(eng, "zlib_sync_64m", torch.from_numpy(np.frombuffer(h, dtype=np.uint8).copy()).cuda(),
                                    d_s, split, args.seconds))
    by = {c["case"]: c for c in out["cases"]}
    if "one_warp_primed_16m" in by:
        base = by["one_warp_primed_16m"]["GBps"]
        out["x_one_warp"] = {c["case"]: round(c["GBps"] / base, 1) for c in out["cases"]
                             if c["case"] != "one_warp_primed_16m"}
    if "primed_mixed_256m" in by and "compat_mixed_256m" in by:
        out["primed_over_compat_mixed"] = round(by["primed_mixed_256m"]["GBps"] / by["compat_mixed_256m"]["GBps"], 3)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
