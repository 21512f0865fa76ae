#!/usr/bin/env python
"""Size-only inflate (zlb_inflate_size_batch) next to the decoder on the same inputs, device resident, plus the
"unknown sizes" case end to end through the host API.

    python tools/bench_inflate_size.py [--seconds S] [--only NAME,...]  -> one JSON line on stdout

Cases (all inputs made from seeds; for every case the size results equal the decoder's field by field):
  bench_inflate_4096x64k  bench.py's inflate leg: synth.mixed(256 MiB, seed 2, segments of 4096) cut into 4096 chunks of
                          64 KiB, each deflated on the GPU (compat mode) into an independent stream; flags 0
  c3_65536x64k            the C3 shape of tools/bench_configs.py: 65 536 streams of 64 KiB, text(65536, 1000 + i) for
                          even i, mixed(65536, 1000 + i) for odd i, 4 GiB of output; made by the GPU compat encoder
                          (whose bytes equal the oracle's RawDeflate, checked by tools/bench_configs.py c3), not by the
                          oracle on the host, which takes minutes of CPU time
  primed_mixed_256m       synth.mixed(256 MiB, 1) in ZLB_MODE_PRIMED, ZLB_INFLATE_SPLIT: split sizing vs the
                          split-window decode (tools/bench_split_window.py)
  zlib_sync_64m           synth.mixed(64 MiB, 3), CPython zlib level 6, a Z_SYNC_FLUSH every 64 KiB, ZLB_INFLATE_SPLIT
  byte_256m               256 MiB of one repeated byte in ZLB_MODE_PRIMED, ZLB_INFLATE_SPLIT
  unknown_sizes_api       16 384 records of 192 KiB (2 KiB of synth.text repeated), through api.py:
                          inflate_many without hints (today's retry loop: 32 KiB, then 128 KiB, then 512 KiB slots --
                          three calls) against inflate_sizes followed by inflate_many(size_hints=...) (two calls);
                          the outputs must be byte-identical
Timing: one warm-up call of each, then size and decode calls alternate until --seconds have passed (at least three of
each) on a host clock; every call ends in a stream synchronise. The per-kernel split comes from one more call of each
with the profile slots on (kernel milliseconds bracketed by CUDA events), not from the timed calls. Rates are
decompressed bytes per second.
"""
import argparse
import json
import os
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np
import torch

import zlibts_b200 as z
from zlibts_b200 import synth
from bench_split_window import deflate_on_gpu, gpu_info

MIB = 1 << 20
FIELDS = ("status", "out_len", "in_used", "blocks")


def chunk_streams(eng, d_in, chunk=65536):
    """Every `chunk` bytes of d_in as an independent stream (GPU compat deflate), packed back to back on the device:
    (packed, items for the decoder)."""
    n = d_in.numel() // chunk
    slot = z.deflate_bound(chunk)
    it = z.make_items(n)
    it["in_off"] = np.arange(n, dtype=np.uint64) * chunk
    it["in_len"], it["out_off"], it["out_cap"] = chunk, np.arange(n, dtype=np.uint64) * slot, slot
    d_slots = torch.empty(n * slot, dtype=torch.uint8, device="cuda")
    r = eng.deflate_batch(d_in, d_slots, it)
    assert int(r["status"].max()) == 0
    lens = r["out_len"].astype(np.uint64)
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64)
    h_slots = d_slots.cpu().numpy()
    del d_slots
    packed = torch.from_numpy(np.concatenate([h_slots[k * slot:k * slot + int(lens[k])] for k in range(n)])).cuda()
    items = z.make_items(n)
    items["in_off"], items["in_len"] = offs, lens
    items["out_off"], items["out_cap"] = np.arange(n, dtype=np.uint64) * chunk, chunk
    return packed, items


def measure(eng, name, d_z, items, d_out, flags, seconds, expect=None):
    out_bytes = int(items["out_cap"].sum())
    sizes = eng.inflate_size_batch(d_z, items, flags)        # warm-up (scratch allocations) and the check
    res = eng.inflate_batch(d_z, d_out, items, flags)
    assert int(res["status"].max()) == 0, name
    for f in FIELDS:
        assert np.array_equal(sizes[f], res[f]), (name, f)
    assert int(sizes["out_len"].sum()) == out_bytes, name
    if expect is not None:
        assert torch.equal(d_out[:expect.numel()], expect), name
    t_size = t_dec = 0.0
    reps = 0
    t_end = time.perf_counter() + seconds
    while reps < 3 or time.perf_counter() < t_end:
        t0 = time.perf_counter()
        eng.inflate_size_batch(d_z, items, flags)
        t1 = time.perf_counter()
        eng.inflate_batch(d_z, d_out, items, flags)
        t2 = time.perf_counter()
        t_size += t1 - t0
        t_dec += t2 - t1
        reps += 1
    kernels = {}
    for what, fn in (("size", lambda: eng.inflate_size_batch(d_z, items, flags)),
                     ("decode", lambda: eng.inflate_batch(d_z, d_out, items, flags))):
        eng.profile_enable(True)
        eng.profile_reset()
        fn()
        prof = eng.profile_read()
        eng.profile_enable(False)
        kernels[what] = {k: {"ms": round(v["ms"], 3), "launches": v["launches"]} for k, v in prof.items() if v["launches"]}
    ms_s, ms_d = t_size * 1e3 / reps, t_dec * 1e3 / reps
    return {"case": name, "items": len(items), "out_bytes": out_bytes, "in_bytes": int(items["in_len"].sum()),
            "flags": flags, "calls_each": reps, "size_ms_per_call": round(ms_s, 3), "decode_ms_per_call": round(ms_d, 3),
            "size_GBps": round(out_bytes / (ms_s * 1e-3) / 1e9, 3), "decode_GBps": round(out_bytes / (ms_d * 1e-3) / 1e9, 3),
            "size_over_decode_speed": round(ms_d / ms_s, 3), "size_faster": ms_s < ms_d,
            "kernels_one_call": kernels, "size_results_equal_decode_results": True}


def single(eng, name, d_plain, d_z, flags, seconds):
    items = z.make_items(1)
    items["in_len"], items["out_cap"] = d_z.numel(), d_plain.numel()
    d_out = torch.empty(d_plain.numel(), dtype=torch.uint8, device="cuda")
    return measure(eng, name, d_z, items, d_out, flags, seconds, d_plain)


def unknown_sizes(seconds):
    recs = []
    for k in range(16384):
        recs.append(np.tile(synth.text(2048, 5000 + k), 96))   # 196 608 bytes, a compression ratio above 20
    bufs, _ = z.deflate_many(recs)
    bufs = [b.copy() for b in bufs]
    ratio = sum(r.size for r in recs) / sum(b.size for b in bufs)
    eng = z.api.engine()
    calls = {"n": 0}
    real = eng.inflate_batch_host

    def counted(*a, **k):
        calls["n"] += 1
        return real(*a, **k)

    eng.inflate_batch_host = counted
    try:
        ref, _ = z.inflate_many(bufs)                          # warm-up
        n_retry = calls["n"]
        sizes = z.inflate_sizes(bufs)
        got, _ = z.inflate_many(bufs, size_hints=sizes)
        n_hinted = calls["n"] - n_retry
        assert all(np.array_equal(a, b) for a, b in zip(ref, got)) and all(np.array_equal(a, r) for a, r in zip(ref, recs))
        t_retry = t_sized = 0.0
        reps = 0
        t_end = time.perf_counter() + seconds
        while reps < 3 or time.perf_counter() < t_end:
            t0 = time.perf_counter()
            a, _ = z.inflate_many(bufs)
            t1 = time.perf_counter()
            s = z.inflate_sizes(bufs)
            b, _ = z.inflate_many(bufs, size_hints=s)
            t2 = time.perf_counter()
            t_retry += t1 - t0
            t_sized += t2 - t1
            reps += 1
        assert all(np.array_equal(x, y) for x, y in zip(a, b))
    finally:
        del eng.inflate_batch_host
    out_bytes = sum(r.size for r in recs)
    ms_r, ms_s = t_retry * 1e3 / reps, t_sized * 1e3 / reps
    return {"case": "unknown_sizes_api", "items": len(recs), "out_bytes": out_bytes, "ratio": round(ratio, 1),
            "retry_loop_decode_calls": n_retry, "sized_decode_calls": n_hinted, "runs_each": reps,
            "retry_loop_ms": round(ms_r, 1), "sizes_then_decode_ms": round(ms_s, 1),
            "retry_loop_GBps": round(out_bytes / (ms_r * 1e-3) / 1e9, 3),
            "sizes_then_decode_GBps": round(out_bytes / (ms_s * 1e-3) / 1e9, 3),
            "sizes_then_decode_faster": ms_s < ms_r, "outputs_identical": True}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=2.0, help="least wall time of the alternating calls per case")
    ap.add_argument("--only", default="", help="comma-separated case names (default: all)")
    args = ap.parse_args()
    only = set(filter(None, args.only.split(",")))
    eng = z.Engine(0)
    z.api.set_engine(eng)
    split = z.INFLATE_SPLIT
    out = {"bench": "inflate_size", **gpu_info(), "cases": []}

    def want(name):
        return not only or name in only

    if want("bench_inflate_4096x64k"):
        d_in = torch.from_numpy(synth.mixed(256 * MIB, 2, 4096)).cuda()
        d_z, items = chunk_streams(eng, d_in)
        d_out = torch.empty(d_in.numel(), dtype=torch.uint8, device="cuda")
        out["cases"].append(measure(eng, "bench_inflate_4096x64k", d_z, items, d_out, 0, args.seconds, d_in))
        del d_in, d_z, d_out
    if want("c3_65536x64k"):
        parts, itemss, at = [], [], 0
        group = 4096
        for g0 in range(0, 65536, group):
            h = np.empty(group * 65536, dtype=np.uint8)
            for k in range(group):
                i = g0 + k
                if i % 2 == 0:
                    synth.text(65536, 1000 + i, out=h[k * 65536:(k + 1) * 65536])
                else:
                    synth.mixed(65536, 1000 + i, 4096, out=h[k * 65536:(k + 1) * 65536])
            d_z, it = chunk_streams(eng, torch.from_numpy(h).cuda())
            it["in_off"] += at
            it["out_off"] += g0 * 65536
            at += d_z.numel()
            parts.append(d_z)
            itemss.append(it)
        d_z = torch.cat(parts)
        del parts
        items = np.concatenate(itemss)
        d_out = torch.empty(65536 * 65536, dtype=torch.uint8, device="cuda")
        out["cases"].append(measure(eng, "c3_65536x64k", d_z, items, d_out, 0, args.seconds))
        del d_z, d_out
    torch.cuda.empty_cache()
    if want("primed_mixed_256m"):
        mixed = torch.from_numpy(synth.mixed(256 * MIB, 1)).cuda()
        out["cases"].append(single(eng, "primed_mixed_256m", mixed, deflate_on_gpu(eng, mixed, z.MODE_PRIMED), split,
                                   args.seconds))
        del mixed
    if want("zlib_sync_64m"):
        h = synth.mixed(64 * MIB, 3).tobytes()
        co = zlib.compressobj(6, zlib.DEFLATED, -15)
        s = b"".join(co.compress(h[k:k + 65536]) + co.flush(zlib.Z_SYNC_FLUSH) for k in range(0, len(h), 65536))
        s += co.flush()
        out["cases"].append(single(eng, "zlib_sync_64m", torch.from_numpy(np.frombuffer(h, dtype=np.uint8).copy()).cuda(),
                                   torch.from_numpy(np.frombuffer(s, dtype=np.uint8).copy()).cuda(), split, args.seconds))
    if want("byte_256m"):
        byte = torch.full((256 * MIB,), 0x61, dtype=torch.uint8, device="cuda")
        out["cases"].append(single(eng, "byte_256m", byte, deflate_on_gpu(eng, byte, z.MODE_PRIMED), split, args.seconds))
        del byte
    torch.cuda.empty_cache()
    if want("unknown_sizes_api"):
        out["cases"].append(unknown_sizes(args.seconds))
    out["size_not_faster"] = [c["case"] for c in out["cases"] if not c.get("size_faster", c.get("sizes_then_decode_faster"))]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
