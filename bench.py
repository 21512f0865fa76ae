#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 DEFLATE engine (BASELINE.json metric / configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--configs all|none|c1,c3,...]
                    [--dump-outputs DIR]

A "step" is one chunk-parallel raw deflate (DYNAMIC blocks, 64 KiB chunks, reference-compatible bytes)
of one 256 MiB `mixed(268435456, seed)` buffer per GPU (SURVEY.md section 8(d), config C2). The same JSON line also
carries: the end-to-end figures through the C-ABI host entry points (page-locked and pageable caller buffers), the
batched-inflate leg (the 4096 independent 64 KiB streams of that buffer), fast / primed modes, an adversarial leg
(2-symbol random, period-3, 8-byte records), and BASELINE's other configs C1, C3, C4, C5 at full size with their
parity checks (`configs`; C5 is sharded over the ranks under --gpus N). Multi-GPU: one process per GPU (torchrun),
every rank owns its own buffer (weak scaling), no data-path collective; the only exchange is the exclusive scan of
the per-rank output sizes.

`--impl reference` times the reference's CPU algorithm (oracle/: C restatement of RawDeflate, pinned to the executed
reference by tests/test_refjs.py; Node is absent from this image) on all host threads over the SAME 256 MiB buffer
per step. That arm neither builds, imports nor loads the CUDA library.
"""
import argparse
import ctypes
import importlib.util
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

CHUNK = 65536
WORKLOAD_BYTES = 256 << 20
METRIC = "deflate_input_GBps"
UNIT = "GB/s"
WORKLOAD = ("C2: 256 MiB mixed(seed=2+rank, seg=4096) per GPU, chunk-parallel raw deflate, 64 KiB chunks, "
            "DYNAMIC blocks, compat mode (bytes == reference RawDeflate per chunk), joined into one stream")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--bytes", type=int, default=WORKLOAD_BYTES, help="per-GPU workload bytes (default = C2)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--configs", default="all", help="BASELINE configs to add to the line: all | none | c1,c3,c4,c5")
    ap.add_argument("--no-extras", action="store_true", help="skip the fast / primed / pageable / adversarial legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; the reference arm keeps none")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _load_py(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", os.environ.get("BENCH_CLOCK_MS", "20")],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        # nvidia-smi needs a moment before its first line: wait for it so that the timed region is covered
        t0 = time.time()
        while self.p is not None and time.time() - t0 < 3.0 and os.path.getsize(self.f.name) == 0:
            time.sleep(0.02)

    def mark(self):
        """call at the start of the timed region: only samples written after this point are reported"""
        self.f.flush()
        self.mark_offset = os.path.getsize(self.f.name)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.05)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()

        def parse(text):
            sm, mx, reasons = [], [], set()
            for line in text.splitlines():
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1]))
                    mx.append(float(c[2]))
                except ValueError:
                    continue
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], c[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, reasons

        self.f.seek(0)
        text = self.f.read()
        off = getattr(self, "mark_offset", 0)
        sm, mx, reasons = parse(text[off:])
        window = "timed region"
        if len(sm) < 2:  # region shorter than two sampling periods: report the whole run under load, say so
            sm, mx, reasons = parse(text)
            window = "warm-up + timed region"
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm),
                       window=window)
        return out


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm (oracle port) on the host cores -- no CUDA library anywhere near it
# ------------------------------------------------------------------------------------------------
def _synth_lib():
    """libzts_synth.so alone (plain C generators of SURVEY Appendix D): built and loaded without the engine."""
    build = _load_py(os.path.join(ROOT, "zlib.ts_b200", "build.py"), "_zts_build")
    build.build_synth()
    lib = ctypes.CDLL(build.SYNTH_LIB)
    lib.zts_gen_mixed.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_uint32]
    return lib


def _mixed_no_engine(n, seed):
    buf = np.empty(n, dtype=np.uint8)
    _synth_lib().zts_gen_mixed(buf.ctypes.data, n, seed & 0xFFFFFFFF, 4096)
    return buf


def cpu_deflate_rate(data, threads, target_s, max_bytes=None):
    """Times oracle RawDeflate per 64 KiB chunk over a bounded prefix sample of `data`.
    Returns (GB/s, sample bytes, compressed bytes of the sample, seconds)."""
    import oracle
    n = len(data)
    probe = min(n, 32 * CHUNK * max(1, threads // 4))
    t0 = time.perf_counter()
    oracle.deflate_chunks_mt(data[:probe], CHUNK, oracle.DYNAMIC, threads)
    dt = max(time.perf_counter() - t0, 1e-4)
    sample = int(min(n, max(probe, probe * target_s / dt)))
    if max_bytes:
        sample = min(sample, max_bytes)
    sample = max(CHUNK, sample // CHUNK * CHUNK)
    t0 = time.perf_counter()
    cbytes = oracle.deflate_chunks_mt(data[:sample], CHUNK, oracle.DYNAMIC, threads)
    dt = time.perf_counter() - t0
    return sample / dt / 1e9, sample, cbytes, dt


def run_reference(args, rank, world):
    if rank != 0:
        return
    import oracle
    oracle.build()
    threads = os.cpu_count() or 1
    n = args.bytes // CHUNK * CHUNK
    data = _mixed_no_engine(n, 2)          # the very buffer rank 0 of the GPU arm compresses
    for _ in range(args.warmup):
        oracle.deflate_chunks_mt(data, CHUNK, oracle.DYNAMIC, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cbytes = oracle.deflate_chunks_mt(data, CHUNK, oracle.DYNAMIC, threads)
    dt = time.perf_counter() - t0
    gbs = n * args.steps / dt / 1e9
    # single-thread figure (north_star: "both single-threaded and across all stated cores")
    st_gbs, st_sample, _, _ = cpu_deflate_rate(data, 1, 3.0)
    sample_txt = f"the whole C2 buffer ({n >> 20} MiB, {n // CHUNK} chunks) per step, {threads} threads"
    line = {
        "impl": "reference", "metric": METRIC, "value": gbs, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD, "bytes_per_gpu": n, "chunk_bytes": CHUNK, "chunks_per_gpu": n // CHUNK,
                   "mode": "compat", "block_type": "DYNAMIC",
                   "note": "reference = C restatement of zlib.ts RawDeflate (oracle/, pinned to the executed reference "
                           "by tests/test_refjs.py); Node is absent from this image; this arm does not load the CUDA library"},
        "ratio": cbytes / n,
        "cpu_baseline": {"value": gbs, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample_txt,
                         "single_thread_value": st_gbs, "single_thread_sample_bytes": st_sample},
        "e2e": {"value": gbs, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def adversarial_inputs(n):
    """SURVEY's worst cases for an exhaustive matcher: 2-symbol random (every 3-byte key has thousands of candidates),
    period-3 ("abcabc..."), 8-byte low-entropy records."""
    rng = np.random.default_rng(20261018)
    r = np.zeros((n // 8, 8), dtype=np.uint8)
    v = (7 * np.arange(n // 8, dtype=np.uint64)).astype(np.uint32)
    for k in range(4):
        r[:, k] = (v >> (8 * k)) & 0xFF
    r[:, 4] = rng.integers(0, 16, n // 8)
    return {"rand2": rng.integers(0, 2, n, dtype=np.uint8), "period3": np.resize(np.frombuffer(b"abc", dtype=np.uint8), n),
            "records8": r.reshape(-1)}


DUMP_SAMPLE = 1 << 22   # stream positions --dump-outputs keeps: 16 MiB of float32 bytes + 32 MiB of float64 indices


def dump_outputs(out_dir, stream, results, rank=0, world=1):
    """--dump-outputs: what the timed deflate call hands its caller, as .npy files under `out_dir`, so that two builds
    can be compared output for output (the inputs are seeded):
      deflate_<field>.npy       every field of the per-item result record (status, crc32, ..., out_len), float64
      deflate_stream.npy        bytes of the compressed stream (uint8 host array `stream`), float32, at the positions
      deflate_stream_index.npy  listed here (float64): every position of a stream of at most DUMP_SAMPLE bytes, else
                                one drawn with a fixed seed from each of DUMP_SAMPLE equal slices of the stream
      deflate_stream_crc32.npy  CRC-32 of the whole stream (float64): covers what the sample skips
    Under --gpus N every rank writes its own files (suffix _rank<r>), sampling DUMP_SAMPLE / N positions: 48 MiB at
    most in all."""
    os.makedirs(out_dir, exist_ok=True)
    sfx = "" if world == 1 else "_rank%d" % rank
    k = DUMP_SAMPLE // world
    if stream.size <= k:
        idx = np.arange(stream.size)
    else:
        edges = np.arange(k + 1, dtype=np.int64) * stream.size // k
        idx = edges[:-1] + (np.random.default_rng(0).random(k) * np.diff(edges)).astype(np.int64)
    arrays = {"stream": stream[idx].astype(np.float32), "stream_index": idx.astype(np.float64),
              "stream_crc32": np.array([zlib.crc32(stream)], dtype=np.float64)}
    arrays.update((f, results[f].astype(np.float64)) for f in results.dtype.names)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, "deflate_%s%s.npy" % (name, sfx)), a)


def run_b200(args, rank, world, local_rank):
    import torch
    import zlibts_b200 as z
    from zlibts_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    z.load_library()
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    n = args.bytes // CHUNK * CHUNK
    n_chunks = n // CHUNK
    data = synth.mixed(n, 2 + rank)
    stream = torch.cuda.Stream()
    eng = z.Engine(local_rank, stream.cuda_stream)
    cap = z.deflate_bound(n)
    cap_primed = z.deflate_bound(n, 0, z.DYNAMIC, z.MODE_PRIMED)   # twice the chunks: larger worst case
    h_in = torch.from_numpy(data).pin_memory()
    h_out = torch.empty(cap, dtype=torch.uint8).pin_memory()
    with torch.cuda.stream(stream):
        d_in = h_in.cuda(non_blocking=True)
        d_out = torch.empty(cap_primed, dtype=torch.uint8, device="cuda")
    stream.synchronize()
    items = z.make_items(1)
    items["in_len"], items["out_cap"] = n, cap

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K calls bracketed by barrier + synchronize; CUDA events on the engine's stream; max over ranks (ms)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        e1.synchronize()
        barrier()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    res = {}

    # every rank but the last leaves its stream open, so the ranks' outputs concatenate into one stream
    dflags = z.DEFLATE_NOT_FINAL if rank < world - 1 else 0

    def step_device():
        res["r"] = eng.deflate_batch(d_in, d_out, items, flags=dflags)

    def step_host():
        res["h"] = eng.deflate_batch_host(h_in, h_out, items, flags=dflags)

    # ---- device-resident leg (value) ---------------------------------------------------------------
    clocks = ClockSampler(local_rank)
    clocks.start()
    for _ in range(args.warmup):
        step_device()
    eng.profile_enable(True)
    eng.profile_reset()
    clocks.mark()
    l0 = eng.launch_count
    ms = timed(step_device, args.steps)
    launches = eng.launch_count - l0
    clk = clocks.stop()
    prof = eng.profile_read()
    eng.profile_enable(False)
    r = res["r"]
    assert int(r["status"][0]) == 0, r
    clen = int(r["out_len"][0])
    value = world * n * args.steps / (ms * 1e-3) / 1e9
    if args.dump_outputs:   # before the legs below reuse d_out
        dump_outputs(args.dump_outputs, d_out[:clen].cpu().numpy(), r, rank, world)

    extras = not args.no_extras
    few = max(1, min(args.steps, 5))
    fast = primed = None
    if extras:
        # ---- fast mode (bounded candidate depth; valid stream, not byte-identical): speed and ratio beside compat ----
        for _ in range(2):
            eng.deflate_batch(d_in, d_out, items, flags=dflags, mode=z.MODE_FAST)
        ms_f = timed(lambda: res.__setitem__("f", eng.deflate_batch(d_in, d_out, items, flags=dflags, mode=z.MODE_FAST)), few)
        fast = {"value": world * n * few / (ms_f * 1e-3) / 1e9, "unit": UNIT, "chain_depth": 16, "steps": few,
                "ratio": int(res["f"]["out_len"][0]) / n, "ratio_vs_compat": int(res["f"]["out_len"][0]) / clen,
                "note": "ratio tolerance vs reference RawDeflate per chunk: 3 % (north_star); compat ratio == reference"}
        # ... with one-step lazy evaluation (ZLB_MODE_LAZY): the ratio falls below the reference's exhaustive greedy parse
        for name, mode in (("lazy_depth16", z.MODE_FAST | z.MODE_LAZY), ("lazy_depth64", z.mode_fast(64) | z.MODE_LAZY)):
            for _ in range(2):
                eng.deflate_batch(d_in, d_out, items, flags=dflags, mode=mode)
            ms_l = timed(lambda: res.__setitem__("l", eng.deflate_batch(d_in, d_out, items, flags=dflags, mode=mode)), few)
            fast[name] = {"value": world * n * few / (ms_l * 1e-3) / 1e9, "unit": UNIT, "steps": few,
                          "ratio": int(res["l"]["out_len"][0]) / n, "ratio_vs_compat": int(res["l"]["out_len"][0]) / clen}
        # ---- primed mode (32 KiB of history in front of every 32 KiB chunk; SURVEY 8(f)-1): ratio recovered, speed paid
        items_p = items.copy()
        items_p["out_cap"] = cap_primed
        primed = {}
        for name, mode in (("exhaustive", z.MODE_PRIMED), ("fast", z.MODE_FAST | z.MODE_PRIMED)):
            for _ in range(2):
                eng.deflate_batch(d_in, d_out, items_p, flags=dflags, mode=mode)
            ms_p = timed(lambda: res.__setitem__("p", eng.deflate_batch(d_in, d_out, items_p, flags=dflags, mode=mode)), few)
            assert int(res["p"]["status"][0]) == 0
            primed[name] = {"value": world * n * few / (ms_p * 1e-3) / 1e9, "unit": UNIT, "steps": few,
                            "ratio": int(res["p"]["out_len"][0]) / n, "ratio_vs_compat": int(res["p"]["out_len"][0]) / clen}
        primed["note"] = ("32 KiB chunks, each searching the 32 KiB before it as well; exhaustive = the reference's matcher "
                          "(blocks equal the oracle's block construction with that history), fast = depth 16")
        step_device()  # leave the compat output in d_out

    # ---- what the host link alone allows: the copies of one step (H2D of the input, D2H of the output, side by side
    #      on two streams, no kernels), every rank at the same time -- the denominator of the end-to-end figures
    def copy_only(h_src, d_dst, d_src, h_dst):
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        def once():
            s1.wait_stream(stream)
            s2.wait_stream(stream)
            with torch.cuda.stream(s1):
                d_dst.copy_(h_src, non_blocking=True)
            with torch.cuda.stream(s2):
                h_dst.copy_(d_src, non_blocking=True)
            stream.wait_stream(s1)
            stream.wait_stream(s2)
        once()
        return timed(once, few) / few
    ms_copy = copy_only(h_in, d_in, d_out[:clen], h_out[:clen])

    # ---- end-to-end leg: host buffers through the C-ABI host entry point (H2D + D2H inside), as many steps as `value`
    for _ in range(max(1, min(2, args.warmup))):
        step_host()
    ms_h = timed(step_host, args.steps)
    assert int(res["h"]["status"][0]) == 0 and int(res["h"]["out_len"][0]) == clen
    e2e_value = world * n * args.steps / (ms_h * 1e-3) / 1e9
    # the same through PAGEABLE caller buffers (what a binding without zlb_host_alloc passes): the library stages them
    e2e_pageable = None
    if extras:
        pg_in, pg_out = data.copy(), np.empty(cap, dtype=np.uint8)
        for _ in range(2):
            eng.deflate_batch_host(pg_in, pg_out, items, flags=dflags)
        ms_pg = timed(lambda: res.__setitem__("hp", eng.deflate_batch_host(pg_in, pg_out, items, flags=dflags)), few)
        assert int(res["hp"]["out_len"][0]) == clen and np.array_equal(pg_out[:clen], h_out.numpy()[:clen])
        e2e_pageable = {"value": world * n * few / (ms_pg * 1e-3) / 1e9, "unit": UNIT, "steps": few,
                        "ms_per_step": ms_pg / few, "ratio_to_pinned": (ms_h / args.steps) / (ms_pg / few),
                        "api": "zlb_deflate_batch_host on pageable numpy buffers (page-locked shadows + copy threads inside)"}
        del pg_in, pg_out

    # ---- inflate leg: the chunks as independent streams (C3-shaped), device resident + host e2e -------
    slot = z.deflate_bound(CHUNK)
    it_c = z.make_items(n_chunks)
    it_c["in_off"] = np.arange(n_chunks, dtype=np.uint64) * CHUNK
    it_c["in_len"] = CHUNK
    it_c["out_off"] = np.arange(n_chunks, dtype=np.uint64) * slot
    it_c["out_cap"] = slot
    with torch.cuda.stream(stream):
        d_slots = torch.empty(n_chunks * slot, dtype=torch.uint8, device="cuda")
    rc = eng.deflate_batch(d_in, d_slots, it_c)
    assert int(rc["status"].max()) == 0
    # pack the streams back to back (what a zip / multi-member container holds)
    lens = rc["out_len"].astype(np.uint64)
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64)
    total_c = int(lens.sum())
    h_slots = d_slots.cpu().numpy()
    h_packed = torch.empty(total_c, dtype=torch.uint8).pin_memory()
    hp = h_packed.numpy()
    for k in range(n_chunks):
        hp[int(offs[k]):int(offs[k] + lens[k])] = h_slots[k * slot:k * slot + int(lens[k])]
    del h_slots, d_slots
    with torch.cuda.stream(stream):
        d_packed = h_packed.cuda(non_blocking=True)
        d_plain = torch.empty(n, dtype=torch.uint8, device="cuda")
    it_i = z.make_items(n_chunks)
    it_i["in_off"], it_i["in_len"] = offs, lens
    it_i["out_off"] = np.arange(n_chunks, dtype=np.uint64) * CHUNK
    it_i["out_cap"] = CHUNK
    h_plain = torch.empty(n, dtype=torch.uint8).pin_memory()

    def inf_device():
        res["i"] = eng.inflate_batch(d_packed, d_plain, it_i)

    def inf_host():
        res["ih"] = eng.inflate_batch_host(h_packed, h_plain, it_i)

    for _ in range(args.warmup):
        inf_device()
    eng.profile_enable(True)
    eng.profile_reset()
    li0 = eng.launch_count
    ms_i = timed(inf_device, args.steps)
    inf_launches = eng.launch_count - li0
    prof_i = eng.profile_read()
    eng.profile_enable(False)
    assert int(res["i"]["status"].max()) == 0
    assert torch.equal(d_plain, d_in), "inflate(deflate(x)) != x"
    inf_value = world * n * args.steps / (ms_i * 1e-3) / 1e9
    inf_host()
    ms_ih = timed(inf_host, args.steps)
    assert torch.equal(h_plain, h_in)
    inf_e2e = world * n * args.steps / (ms_ih * 1e-3) / 1e9
    ms_icopy = copy_only(h_packed, d_packed, d_plain, h_plain)
    inf_pageable = None
    if extras:
        pg_c, pg_p = h_packed.numpy().copy(), np.empty(n, dtype=np.uint8)
        for _ in range(2):
            eng.inflate_batch_host(pg_c, pg_p, it_i)
        ms_ipg = timed(lambda: eng.inflate_batch_host(pg_c, pg_p, it_i), few)
        assert np.array_equal(pg_p, data)
        inf_pageable = {"value": world * n * few / (ms_ipg * 1e-3) / 1e9, "unit": UNIT, "steps": few,
                        "ms_per_step": ms_ipg / few, "ratio_to_pinned": (ms_ih / args.steps) / (ms_ipg / few)}
        del pg_c, pg_p

    # ---- the one cross-rank exchange: exclusive scan of the per-rank output sizes ----------------------
    rank_off = 0
    if dist is not None:
        sizes = torch.zeros(world, dtype=torch.int64, device="cuda")
        sizes[rank] = clen
        dist.all_reduce(sizes)
        rank_off = int(sizes[:rank].sum().item())
        total_clen = int(sizes.sum().item())
    else:
        total_clen = clen

    # ---- roofline of the dominant kernel -------------------------------------------------------------
    peak, peak_src = peaks()
    top = max(prof.items(), key=lambda kv: kv[1]["ms"])
    top_name, top_ms, top_launches = top[0], top[1]["ms"], top[1]["launches"]
    step_kernel_ms = sum(v["ms"] for v in prof.values())
    alg_bytes_per_step = n + clen                      # SURVEY 8(d): N + C per chunk, summed over the step's chunks
    alg_bytes_per_launch = alg_bytes_per_step * args.steps / max(1, top_launches)
    avg_launch_ms = top_ms / max(1, top_launches)
    achieved = alg_bytes_per_launch / (avg_launch_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": top_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes_per_launch, "avg_launch_ms": avg_launch_ms,
                "kernel_share_of_step": top_ms / max(step_kernel_ms, 1e-9),
                "kernels_ms_per_step": {k: v["ms"] / args.steps for k, v in prof.items() if v["launches"]},
                "note": "the kernel is issue-bound, not HBM-bound: see issue_frac"}
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file):
        try:
            tj = json.load(open(traffic_file))
            units = n_chunks * args.steps / max(1, top_launches)   # chunks per launch of this run
            per_unit = tj.get(top_name, 0) / max(1, tj.get("_units_per_launch", 1))
            roofline["traffic"] = per_unit * units or None
            roofline["traffic_source"] = "carried from profiles/ (not measured in this run): " + str(tj.get("_note"))
            inst = tj.get("_inst_executed", {}).get(top_name)
            if inst and clk.get("sm_mhz"):
                # warp instructions issued / issue slots of the device during the launch (4 schedulers per SM, 1 per clock)
                sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
                per_launch = inst / max(1, tj.get("_units_per_launch", 1)) * units
                slots = sm_count * 4 * clk["sm_mhz"] * 1e6 * avg_launch_ms * 1e-3
                roofline["issue_frac"] = per_launch / slots
                roofline["warp_instructions_per_input_byte"] = per_launch / (n * args.steps / max(1, top_launches))
                roofline["issue_frac_source"] = "smsp__inst_executed.sum carried from profiles/ (ncu), clocks and time of this run"
        except Exception:
            pass
    inf_top_ms = prof_i["inflate_warp_kernel"]["ms"] / max(1, prof_i["inflate_warp_kernel"]["launches"])
    inf_roofline = {"bound": "hbm", "kernel": "inflate_warp_kernel",
                    "achieved": (n + total_c) / (inf_top_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s"}
    inf_roofline["frac"] = inf_roofline["achieved"] / peak

    # ---- adversarial inputs (rank 0, N = 1): throughput on 64 MiB of each and the time of ONE chunk --------------
    adversarial = None
    if extras and rank == 0 and world == 1:
        adversarial = {}
        an = 64 << 20
        it_a = z.make_items(1)
        it_a["in_len"], it_a["out_cap"] = an, z.deflate_bound(an)
        it_1 = z.make_items(1)
        it_1["in_len"], it_1["out_cap"] = CHUNK, z.deflate_bound(CHUNK)
        for name, arr in adversarial_inputs(an).items():
            with torch.cuda.stream(stream):
                d_a = torch.from_numpy(np.ascontiguousarray(arr)).cuda()
            for _ in range(2):
                ra = eng.deflate_batch(d_a, d_out, it_a)
            ms_a = timed(lambda: eng.deflate_batch(d_a, d_out, it_a), 3)
            eng.deflate_batch(d_a, d_out, it_1)
            ms_1 = timed(lambda: eng.deflate_batch(d_a, d_out, it_1), 5)
            adversarial[name] = {"value": an * 3 / (ms_a * 1e-3) / 1e9, "unit": UNIT, "ratio": int(ra["out_len"][0]) / an,
                                 "one_chunk_ms": ms_1 / 5}
            del d_a
        adversarial["note"] = ("64 MiB each, compat mode; one_chunk_ms = a single 64 KiB chunk through the whole pipeline "
                               "(one CTA): what the slowest chunk of a wave can cost")

    # ---- CPU baseline beside it (rank 0, N = 1 only): oracle port on a bounded sample ------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import oracle
        oracle.build()
        threads = os.cpu_count() or 1
        gbs, sample, cbytes, secs = cpu_deflate_rate(data, threads, args.cpu_seconds, max_bytes=n)
        st_gbs, _, _, _ = cpu_deflate_rate(data, 1, 3.0)
        # the sample doubles as a parity check: compat bytes => identical sizes for those chunks
        gpu_sample = int(rc["out_len"][: sample // CHUNK].sum())
        cpu = {"value": gbs, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"first {sample >> 20} MiB of the C2 buffer ({sample // CHUNK} chunks), {secs:.1f} s, "
                         f"{threads} threads; C restatement of reference RawDeflate (Node absent)",
               "single_thread_value": st_gbs, "sample_ratio": cbytes / sample,
               "gpu_bytes_equal_on_sample": bool(gpu_sample == cbytes)}

    # ---- BASELINE's other configs at full size, with their parity checks ------------------------------------------
    configs = None
    want = [] if args.configs == "none" else (["c1", "c3", "c4", "c5"] if args.configs == "all" else args.configs.split(","))
    if want:
        del d_packed, d_plain, h_plain
        torch.cuda.empty_cache()
        bc = _load_py(os.path.join(ROOT, "tools", "bench_configs.py"), "_bench_configs")
        configs = {}
        for name in want:
            try:
                if name == "c5":
                    configs["c5"] = bc.c5_sharded(eng, stream, rank, world, dist)    # every rank takes part
                elif rank == 0 and world == 1:
                    configs[name] = getattr(bc, name)(eng)
            except Exception as e:  # a config that cannot run here (host memory, ...) must not take the headline down
                configs[name] = {"error": repr(e)[:300]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "bytes_per_gpu": n, "chunk_bytes": CHUNK, "chunks_per_gpu": n_chunks,
                       "mode": "compat", "block_type": "DYNAMIC", "parallelism": f"shard{world}",
                       "l2": "inputs (256 MiB) larger than L2 (126 MB), no flush",
                       "timers": "value: CUDA events around K calls with the per-kernel event timers on (they feed roofline)"},
            "ratio": clen / n,
            "fast_mode": fast,
            "primed_mode": primed,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n, "d2h_bytes_per_step": clen,
                    "ms_per_step": ms_h / args.steps, "steps": args.steps,
                    "api": "zlb_deflate_batch_host (page-locked host buffers)",
                    "copies_alone_ms": ms_copy, "copies_alone_value": world * n / (ms_copy * 1e-3) / 1e9,
                    "frac_of_copies_alone": ms_copy / (ms_h / args.steps),
                    "copies_alone_note": "H2D of the input and D2H of the output of one step on two streams, no kernels, "
                                         "all ranks at once, max over ranks: the host link's ceiling for this leg"},
            "e2e_pageable": e2e_pageable,
            "gpu_launches": int(launches),
            "clocks": {"sm_mhz": clk["sm_mhz"], "sm_max_mhz": clk["sm_max_mhz"], "reasons": clk["reasons"],
                       "samples": clk["samples"], "window": clk.get("window")},
            "roofline": roofline,
            "cpu_baseline": cpu,
            "inflate": {"metric": "inflate_output_GBps", "value": inf_value, "unit": UNIT, "streams_per_gpu": n_chunks,
                        "ms_per_step": ms_i / args.steps, "gpu_launches": int(inf_launches),
                        "e2e": {"value": inf_e2e, "unit": UNIT, "h2d_bytes_per_step": total_c,
                                "d2h_bytes_per_step": n, "ms_per_step": ms_ih / args.steps, "steps": args.steps,
                                "copies_alone_ms": ms_icopy, "copies_alone_value": world * n / (ms_icopy * 1e-3) / 1e9,
                                "frac_of_copies_alone": ms_icopy / (ms_ih / args.steps)},
                        "e2e_pageable": inf_pageable,
                        "roofline": inf_roofline},
            "adversarial": adversarial,
            "configs": configs,
            "multi_gpu": {"output_bytes_total": total_clen, "rank0_offset": rank_off,
                          "exchange": "exclusive scan of per-rank output sizes (8-byte all-reduce), no data-path collective"},
        }
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """The one JSON line goes to the real stdout; everything else the libraries print (NCCL banner, ...) was
    redirected to stderr at start-up so that stdout carries exactly one line."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)   # builds the oracle and the generators only; never touches the CUDA library
        return
    import __graft_entry__ as g
    if rank == 0 or not os.path.exists(os.path.join(ROOT, "zlib.ts_b200", "libzlibts_b200.so")):
        g.build()
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
