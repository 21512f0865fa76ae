"""Random access through an index of access points (zlb_inflate_index / zlb_inflate_ranges) on the GPU.

Measures, with the card's name and power limit read in the same run:
  * the index build against the plain ZLB_INFLATE_SPLIT decode of the same stream (256 MiB through this engine's
    compat mode, 256 MiB of mixed and of text through CPython zlib -6, 16 MiB through Z_FIXED);
  * a whole-stream read through the index at 64 KiB / 256 KiB / 1 MiB spacing against the SPLIT decode (a read is cut
    at every point, so its parallelism is size / spacing warps);
  * batches of 4096 random 4 KiB and 64 KiB reads over a 1 GiB zlib -6 stream at each spacing: reads per second with
    the data on the device, and through api.read_ranges (host buffers, the compressed stream copied over per call);
  * the index's size.
Times are host clocks around calls that end in a device synchronise, median of --reps runs after one warm-up.

    python tools/bench_inflate_index.py [--out profiles/r03e_inflate_index.json] [--reps 3] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
MIB = 1 << 20


def _card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def _median(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t)
    return float(np.median(ts))


def _raw(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    return co.compress(data) + co.flush()


class Stream:
    def __init__(self, eng, name, comp, size):
        import torch
        import zlibts_b200 as z
        self.eng, self.name, self.size = eng, name, size
        self.d_in = torch.from_numpy(np.frombuffer(comp, dtype=np.uint8).copy()).cuda()
        self.d_out = torch.empty(max(size, 1), dtype=torch.uint8, device="cuda")
        self.items = z.make_items(1)
        self.items["in_len"], self.items["out_cap"] = len(comp), size
        self.comp_len = len(comp)

    def split(self):
        import zlibts_b200 as z
        r = self.eng.inflate_batch(self.d_in, self.d_out, self.items, z.INFLATE_SPLIT)
        assert int(r["status"][0]) == 0 and int(r["out_len"][0]) == self.size

    def index(self, spacing):
        r, p, c = self.eng.inflate_index(self.d_in, self.d_out, self.items, [0, self.size // spacing + 2], spacing)
        assert int(r["status"][0]) == 0
        return p[:int(c[0])].copy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03e_inflate_index.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    import torch
    import zlibts_b200 as z
    from zlibts_b200 import synth
    eng = z.Engine(0)
    z.api.set_engine(eng)
    big = 16 * MIB if args.quick else 256 * MIB
    huge = 32 * MIB if args.quick else 1024 * MIB
    out = {"card": _card(), "reps": args.reps, "timing": "host clock around synchronising calls, median",
           "build": [], "whole_read": [], "random_reads": []}
    spacings = (64 << 10, 256 << 10, 1 << 20)

    # ---- build against the SPLIT decode
    mixed, text = synth.mixed(big, 301).tobytes(), synth.text(big, 302).tobytes()
    cases = [("compat_mixed", None, mixed), ("zlib6_mixed", _raw(mixed, 6), mixed), ("zlib6_text", _raw(text, 6), text),
             ("zfixed_text_16MiB", _raw(text[:16 * MIB], 6, zlib.Z_FIXED), text[:16 * MIB])]
    for name, comp, data in cases:
        if comp is None:
            d = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).cuda()
            cap = z.deflate_bound(len(data))
            d_z = torch.empty(cap, dtype=torch.uint8, device="cuda")
            it = z.make_items(1)
            it["in_len"], it["out_cap"] = len(data), cap
            r = eng.deflate_batch(d, d_z, it)
            comp = d_z[:int(r["out_len"][0])].cpu().numpy().tobytes()
            del d, d_z
        s = Stream(eng, name, comp, len(data))
        t_split = _median(s.split, args.reps)
        row = {"stream": name, "bytes": len(data), "compressed": len(comp), "split_s": t_split,
               "split_GBps": len(data) / t_split / 1e9}
        for sp in spacings:
            t = _median(lambda: s.index(sp), args.reps)
            row["index_s_%dK" % (sp >> 10)] = t
            row["points_%dK" % (sp >> 10)] = len(s.index(sp))
        assert s.d_out.cpu().numpy().tobytes() == data
        out["build"].append(row)
        print(json.dumps(row), flush=True)
        # ---- a whole-stream read through the index against the split
        if name == "zlib6_mixed":
            for sp in spacings:
                pts = s.index(sp)
                rg = z.make_ranges(1)
                rg[0] = (0, s.comp_len, 0, len(pts), 0, 0, s.size)
                d_o = torch.empty_like(s.d_out)
                t = _median(lambda: eng.inflate_ranges(s.d_in, s.d_out, d_o, pts, rg), args.reps)
                assert d_o.cpu().numpy().tobytes() == data
                row = {"stream": name, "spacing": sp, "points": len(pts), "read_s": t, "read_GBps": s.size / t / 1e9,
                       "split_s": t_split}
                out["whole_read"].append(row)
                print(json.dumps(row), flush=True)
        del s
        torch.cuda.empty_cache()

    # ---- random reads over a large zlib -6 stream
    data = synth.text(huge, 303).tobytes()
    comp = zlib.compress(data, 6)
    rng = np.random.default_rng(304)
    for sp in spacings:
        ref, idx = z.inflate_index(comp, "zlib", spacing=sp)
        assert ref.tobytes() == data
        s = Stream(eng, "zlib6_text_%dMiB" % (huge >> 20), comp[2:], len(data))
        pts = idx.points.copy()
        d_win = torch.from_numpy(idx.windows.copy()).cuda()
        for ln in (4096, 65536):
            n = 4096
            pos = rng.integers(0, len(data) - ln, n)
            rg = z.make_ranges(n)
            rg["in_len"], rg["pt_count"], rg["pos"] = s.comp_len, len(pts), pos
            rg["out_off"], rg["out_cap"] = np.arange(n, dtype=np.uint64) * ln, ln
            d_o = torch.empty(n * ln, dtype=torch.uint8, device="cuda")
            t_dev = _median(lambda: eng.inflate_ranges(s.d_in, d_win, d_o, pts, rg), args.reps)
            o = d_o.cpu().numpy()
            for k in range(0, n, 97):
                assert o[k * ln:(k + 1) * ln].tobytes() == data[int(pos[k]):int(pos[k]) + ln]
            spans = [(int(p), ln) for p in pos]
            t_api = _median(lambda: idx.read_many(comp, spans), args.reps)
            row = {"stream": s.name, "spacing": sp, "points": len(idx), "index_bytes": idx.nbytes, "reads": n,
                   "read_bytes": ln, "device_s": t_dev, "device_reads_per_s": n / t_dev, "api_s": t_api,
                   "api_reads_per_s": n / t_api}
            out["random_reads"].append(row)
            print(json.dumps(row), flush=True)
        del s, d_win
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
