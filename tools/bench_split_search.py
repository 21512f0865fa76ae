#!/usr/bin/env python
"""Chunk-parallel inflate of streams without sync-flush markers (ZLB_INFLATE_SPLIT, searched cuts), device resident.

    python tools/bench_split_search.py [--seconds S] [--only NAME,...]  -> one JSON line on stdout

Cases (all inputs made from seeds; every output is compared with the input):
  zlib6_text_256m      synth.text(256 MiB, 2) through CPython zlib level 6, raw deflate, no flushes
  zlib6_mixed_256m     synth.mixed(256 MiB, 1), the same
  zlib1_mixed_256m     the same data at level 1
  zlib9_mixed_256m     the same data at level 9
  random6_256m         256 MiB of random bytes at level 6: stored blocks, cut through stored candidates
  gunzip_gzip6_256m    GUnzip(gzip.compress(mixed, 6)).decompress() through api.py, host bytes in and out (end to end)
  fixed_16m            synth.mixed(16 MiB, 1) at level 6 with Z_FIXED: no candidates, the cost of a failed search
                       beside the one-warp route on the same stream (fixed_16m_one_warp)
  one_warp_zlib6_16m   synth.mixed(16 MiB, 1) at level 6 without ZLB_INFLATE_SPLIT: what such streams got before
  primed_mixed_256m,   the r03a cases: a GPU primed stream (window mode) and a GPU compat stream (independent pieces)
  compat_mixed_256m    of synth.mixed(256 MiB, 1), as a check that the marker route is unchanged
Each device case also reports the per-kernel split of one call with the profile slots on (kernel milliseconds
bracketed by CUDA events: block_find_kernel is the finder, inflate_warp_kernel_size the size pass and its repair
rounds). The number of pieces of a searched case is about the finder's distinct proposals at the split's 32 KiB
step (`finder_step`; cuts closer than 64 bytes and repairs are not counted there).
`finder_step` runs the finder alone (zlb_debug_block_starts) on the zlib6_text / zlib6_mixed streams with nominal cuts
every 16, 32 and 64 KiB, as the split lays them out: kernel milliseconds and the distinct block starts it proposes.
Timing: one warm-up call, then as many calls as fit in --seconds (at least two) on a host clock; zlb_inflate_batch
ends in a stream synchronise. Outputs of 256 MiB do not fit the 126 MB L2.
"""
import argparse
import gzip
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


def raw(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    return co.compress(data) + co.flush()


def dev(b):
    return torch.from_numpy(np.frombuffer(b, dtype=np.uint8).copy()).cuda()


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


def finder_step(eng, name, s):
    """the finder alone with nominal cuts every 16 / 32 / 64 KiB over the whole stream"""
    d_s = dev(s)
    out = {"case": name, "in_bytes": len(s)}
    for step in (16 << 10, 32 << 10, 64 << 10):
        cuts = np.arange(step, len(s), step, dtype=np.uint64)
        eng.debug_block_starts(d_s, cuts, 8 * step)  # warm-up
        eng.profile_enable(True)
        eng.profile_reset()
        got = eng.debug_block_starts(d_s, cuts, 8 * step)
        prof = eng.profile_read()
        eng.profile_enable(False)
        out["step_%dk" % (step >> 10)] = {"cuts": len(cuts), "distinct_starts": int(len(set(got[got >= 0].tolist()))),
                                          "finder_ms": round(prof["block_find_kernel"]["ms"], 3)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0, help="least wall time of the timed calls per case")
    ap.add_argument("--only", default="", help="comma-separated case names (default: all)")
    args = ap.parse_args()
    only = set(filter(None, args.only.split(",")))
    eng = z.Engine(0)
    split = z.INFLATE_SPLIT
    out = {"bench": "split_search", **gpu_info(), "cases": [], "finder_step": []}

    def want(name):
        return not only or name in only

    mixed_h = synth.mixed(256 * MIB, 1).tobytes()
    mixed = dev(mixed_h)
    for level in (6, 1, 9):
        name = "zlib%d_mixed_256m" % level
        if want(name):
            s = raw(mixed_h, level)
            out["cases"].append(measure(eng, name, mixed, dev(s), split, args.seconds))
            if level == 6:
                out["finder_step"].append(finder_step(eng, name, s))
    if want("gunzip_gzip6_256m"):
        g = gzip.compress(mixed_h, 6)
        z.api.set_engine(eng)
        assert z.GUnzip(g).decompress().tobytes() == mixed_h
        reps, t0 = 0, time.perf_counter()
        while True:
            o = z.GUnzip(g).decompress()
            reps += 1
            el = time.perf_counter() - t0
            if reps >= 2 and el >= args.seconds:
                break
        assert o.tobytes() == mixed_h
        ms = el * 1e3 / reps
        out["cases"].append({"case": "gunzip_gzip6_256m", "out_bytes": len(mixed_h), "in_bytes": len(g),
                             "ms_per_call": round(ms, 3), "GBps": round(len(mixed_h) / (ms * 1e-3) / 1e9, 3),
                             "calls": reps, "end_to_end_host_bytes": True, "output_equals_input": True})
        del g
    m16_h = mixed_h[:16 * MIB]
    m16 = dev(m16_h)
    if want("fixed_16m"):
        s = dev(raw(m16_h, 6, zlib.Z_FIXED))
        out["cases"].append(measure(eng, "fixed_16m", m16, s, split, args.seconds))
        out["cases"].append(measure(eng, "fixed_16m_one_warp", m16, s, 0, 0.0))
    if want("one_warp_zlib6_16m"):
        out["cases"].append(measure(eng, "one_warp_zlib6_16m", m16, dev(raw(m16_h, 6)), 0, 0.0))
    if want("primed_mixed_256m"):
        out["cases"].append(measure(eng, "primed_mixed_256m", mixed, deflate_on_gpu(eng, mixed, z.MODE_PRIMED), split,
                                    args.seconds))
    if want("compat_mixed_256m"):
        out["cases"].append(measure(eng, "compat_mixed_256m", mixed, deflate_on_gpu(eng, mixed, z.MODE_COMPAT), split,
                                    args.seconds))
    del mixed, mixed_h
    if want("zlib6_text_256m"):
        text_h = synth.text(256 * MIB, 2).tobytes()
        s = raw(text_h, 6)
        out["cases"].append(measure(eng, "zlib6_text_256m", dev(text_h), dev(s), split, args.seconds))
        out["finder_step"].append(finder_step(eng, "zlib6_text_256m", s))
        del text_h, s
    if want("random6_256m"):
        r_h = np.random.default_rng(5).integers(0, 256, 256 * MIB, dtype=np.uint8).tobytes()
        out["cases"].append(measure(eng, "random6_256m", dev(r_h), dev(raw(r_h, 6)), split, args.seconds))
    for c in out["cases"]:
        k = c.get("kernels_one_call", {})
        if "inflate_warp_kernel_window" in k and "block_find_kernel" in k:
            c["size_pass_ms"] = k.get("inflate_warp_kernel_size", {}).get("ms")
            c["finder_ms"] = k["block_find_kernel"]["ms"]
    by = {c["case"]: c for c in out["cases"]}
    if "one_warp_zlib6_16m" in by:
        base = by["one_warp_zlib6_16m"]["GBps"]
        out["x_one_warp"] = {c["case"]: round(c["GBps"] / base, 1) for c in out["cases"]
                             if c["case"] != "one_warp_zlib6_16m"}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
