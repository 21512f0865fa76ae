#!/usr/bin/env python
"""Preset dictionaries (zlb_deflate_batch_dict / zlb_inflate_batch_dict), device resident.

    python tools/bench_dictionary.py [--records N] [--seconds S] [--out FILE]  -> one JSON line on stdout (and FILE)

Inputs (made from seeds): N records (default 65536) of 256 B .. 4 KiB, consecutive slices of synth.text(seed 31),
about 140 MB in all -- more than the 126 MB L2. The dictionaries are 4 KiB and 32 KiB of other records of the same
generator (the text behind the records), shared by every record.
Reported:
  ratio           compressed / input bytes: the GPU's compat mode without and with each dictionary, and CPython zlib
                  level 6 with the same zdict (raw deflate, one compressobj per record)
  deflate, inflate  GB/s per input (deflate) / output (inflate) byte of one batched call of all records, with and
                  without each dictionary; one warm-up call, then calls for --seconds on a host clock (every call ends
                  in a stream synchronise); every output is checked
  split_256m      one 256 MiB synth.text stream deflated in primed mode with the 32 KiB dictionary, inflated with
                  ZLB_INFLATE_SPLIT (the window route starts from the dictionary), and the kernels one call ran; the
                  same stream deflated without a dictionary, for comparison
The card's name and power limit are read in the same run.
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


def timed(fn, seconds):
    fn()  # warm-up: scratch allocations
    reps, t0 = 0, time.perf_counter()
    while True:
        fn()
        reps += 1
        el = time.perf_counter() - t0
        if reps >= 2 and el >= seconds:
            return el * 1e3 / reps, reps


def dict_table(n, dictionary):
    t = z.make_dicts(n)
    if dictionary is not None:
        t["len"] = len(dictionary)
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=65536)
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    eng = z.Engine(0)
    rng = np.random.default_rng(31)
    lens = rng.integers(256, 4097, args.records).astype(np.uint64)
    total = int(lens.sum())
    src = synth.text(total + 64 * 1024, 31).tobytes()
    recs_blob = np.frombuffer(src[:total], dtype=np.uint8).copy()
    dicts = {"none": None, "4k": src[total:total + 4096], "32k": src[total + 4096:total + 4096 + 32768]}
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64)
    d_in = torch.from_numpy(recs_blob).cuda()
    out = {"bench": "dictionary", **gpu_info(), "records": args.records, "input_bytes": total, "cases": []}

    for name, dd in dicts.items():
        table = dict_table(args.records, dd)
        d_dict = torch.from_numpy(np.frombuffer(dd or b"\0", dtype=np.uint8).copy()).cuda()
        caps = np.array([z.deflate_bound(int(n), 0, z.DYNAMIC, 0, dd is not None) for n in lens], dtype=np.uint64)
        ooffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.uint64)
        items = z.make_items(args.records)
        items["in_off"], items["in_len"], items["out_off"], items["out_cap"] = offs, lens, ooffs[:-1], caps
        d_z = torch.empty(int(ooffs[-1]), dtype=torch.uint8, device="cuda")
        res = [None]

        def defl():
            res[0] = eng.deflate_batch(d_in, d_z, items, d_dict=d_dict, dicts=table)
        ms_d, reps_d = timed(defl, args.seconds)
        r = res[0]
        assert int(r["status"].max()) == 0
        comp = int(r["out_len"].sum())
        # inflate of what was just written, back into a zeroed buffer; checked against the input
        iitems = z.make_items(args.records)
        iitems["in_off"], iitems["in_len"] = ooffs[:-1], r["out_len"]
        iitems["out_off"], iitems["out_cap"] = offs, lens
        d_back = torch.zeros(total, dtype=torch.uint8, device="cuda")

        def infl():
            res[0] = eng.inflate_batch(d_z, d_back, iitems, 0, d_dict, table)
        ms_i, reps_i = timed(infl, args.seconds)
        assert int(res[0]["status"].max()) == 0 and torch.equal(d_back, d_in), name
        # CPython zlib level 6 with the same zdict, record by record
        cpy = 0
        for o, n in zip(offs.tolist(), lens.tolist()):
            co = zlib.compressobj(6, zlib.DEFLATED, -15, 9, zlib.Z_DEFAULT_STRATEGY, **({"zdict": dd} if dd else {}))
            cpy += len(co.compress(src[o:o + n]) + co.flush())
        out["cases"].append({
            "dictionary": name, "dictionary_bytes": len(dd or b""),
            "ratio_gpu_compat": round(comp / total, 4), "ratio_cpython_level6": round(cpy / total, 4),
            "deflate_ms": round(ms_d, 3), "deflate_GBps": round(total / (ms_d * 1e-3) / 1e9, 3), "deflate_calls": reps_d,
            "inflate_ms": round(ms_i, 3), "inflate_GBps": round(total / (ms_i * 1e-3) / 1e9, 3), "inflate_calls": reps_i,
            "output_equals_input": True})
        del d_z, d_back

    # one 256 MiB stream, primed mode, with the 32 KiB dictionary (the split route's window mode starts from it) and,
    # for comparison, without one
    big = synth.text(256 * MIB, 32)
    d_big = torch.from_numpy(big).cuda()
    d_o = torch.zeros(d_big.numel(), dtype=torch.uint8, device="cuda")
    out["split_256m"] = {}
    for label, dd in (("dictionary_32k", dicts["32k"]), ("no_dictionary", None)):
        d_dict = torch.from_numpy(np.frombuffer(dd or b"\0", dtype=np.uint8).copy()).cuda()
        table = dict_table(1, dd)
        cap = z.deflate_bound(d_big.numel(), 0, z.DYNAMIC, z.MODE_PRIMED, dd is not None)
        it = z.make_items(1)
        it["in_len"], it["out_cap"] = d_big.numel(), cap
        d_z = torch.empty(cap, dtype=torch.uint8, device="cuda")
        r = eng.deflate_batch(d_big, d_z, it, mode=z.MODE_PRIMED, d_dict=d_dict, dicts=table)
        assert int(r["status"][0]) == 0
        clen = int(r["out_len"][0])
        it2 = z.make_items(1)
        it2["in_len"], it2["out_cap"] = clen, d_big.numel()

        def run():
            r2 = eng.inflate_batch(d_z, d_o, it2, z.INFLATE_SPLIT, d_dict, table)
            assert int(r2["status"][0]) == 0
        ms, reps = timed(run, args.seconds)
        assert torch.equal(d_o, d_big), label
        eng.profile_enable(True)
        eng.profile_reset()
        run()
        prof = eng.profile_read()
        eng.profile_enable(False)
        out["split_256m"][label] = {
            "out_bytes": d_big.numel(), "in_bytes": clen, "dictionary_bytes": len(dd or b""),
            "ms_per_call": round(ms, 3), "GBps": round(d_big.numel() / (ms * 1e-3) / 1e9, 3), "calls": reps,
            "kernels_one_call": {k: {"ms": round(v["ms"], 3), "launches": v["launches"]}
                                 for k, v in prof.items() if v["launches"]},
            "output_equals_input": True}
        d_o.zero_()
        del d_z
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
