"""GPU: the "_host" deflate entry point against the device entry point, on every route: stored, fixed and dynamic
blocks, the primed, fast and smallest modes, preset dictionaries and checksums. The batch sizes take each way the
outputs come back to the host: per wave (at most 256 items), merged runs, and the span with the slack zeroed on the
device (more than 2048 runs). Every call goes through page-locked and through pageable buffers."""
import functools
import zlib

import numpy as np
import pytest

import oracle
from helpers import pack, rand_bytes

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5


@functools.lru_cache(maxsize=None)
def _inputs(n, seed):
    """n seeded inputs of 1 to 3000 bytes, from two symbols to random bytes."""
    rng = np.random.default_rng(seed)
    sizes, alphabets = rng.integers(1, 3001, n), rng.choice([2, 4, 26, 256], n)
    return tuple(rand_bytes(rng, int(k), int(a)).tobytes() for k, a in zip(sizes, alphabets))


def test_many_stored_items_come_back_through_the_host_entry_point(engine):
    """3000 stored items: more than 2048 copies, so the copy-back zeroes every slot's slack on the device by the
    device's results and copies one span. The stored route's results must be on the device like every other route's
    (with zeros there, every body came back zeroed)."""
    import zlibts_b200 as z
    z.api.set_engine(engine)
    datas = _inputs(3000, 41)
    outs, res = z.api.deflate_many(datas, z.api.CompressionType.NONE, want_crc32=True)
    for d, o, r in zip(datas, outs, res):
        o = o.tobytes()
        assert int(r["status"]) == 0
        assert o == oracle.raw_deflate(d, oracle.NONE)
        assert zlib.decompress(o, -15) == d
        assert int(r["crc32"]) == zlib.crc32(d)


# route: (block type, mode, chunk bytes, preset dictionaries)
ROUTES = {
    "stored": (oracle.NONE, 0, 0, False),
    "fixed": (oracle.FIXED, 0, 256, False),        # small chunks: several waves on two streams
    "dynamic": (oracle.DYNAMIC, 0, 0, False),
    "primed": (oracle.DYNAMIC, "MODE_PRIMED", 1024, False),
    "fast": (oracle.DYNAMIC, "MODE_FAST", 0, False),
    "smallest": (oracle.DYNAMIC, "MODE_SMALLEST", 0, False),
    "dictionary": (oracle.DYNAMIC, 0, 0, True),
}
FLAGS = {"plain": (), "sums": ("DEFLATE_WANT_CRC32", "DEFLATE_WANT_ADLER32"),
         "sums_not_final": ("DEFLATE_WANT_CRC32", "DEFLATE_WANT_ADLER32", "DEFLATE_NOT_FINAL")}


@pytest.mark.parametrize("flags_name", list(FLAGS))
@pytest.mark.parametrize("route", list(ROUTES))
def test_host_entry_point_equals_the_device_entry_point(engine, route, flags_name):
    import torch
    import zlibts_b200 as z
    block_type, mode, chunk, with_dict = ROUTES[route]
    mode = getattr(z, mode) if mode else z.MODE_COMPAT
    flags = 0
    for f in FLAGS[flags_name]:
        flags |= getattr(z, f)
    for n in (200, 600, 3000):
        datas = _inputs(n, n)
        blob, offs, lens = pack(datas)
        rng = np.random.default_rng(n + 1)
        dicts = h_dict = d_dict = None
        if with_dict:  # none, 100 bytes or 32 KiB, in turn
            h_dict = rand_bytes(rng, 100 + 32768, 26)
            d_dict = torch.from_numpy(h_dict).cuda()
            dicts = z.make_dicts(n)
            dicts["off"][2::3] = 100
            dicts["len"][1::3], dicts["len"][2::3] = 100, 32768
        caps = [z.deflate_bound(k, chunk, block_type, mode, with_dict) for k in lens]
        ooffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.uint64)
        items = z.make_items(n)
        items["in_off"], items["in_len"], items["out_off"], items["out_cap"] = offs, lens, ooffs[:-1], caps
        total = int(ooffs[-1])
        d_out = torch.zeros(total, dtype=torch.uint8, device="cuda")
        rd = engine.deflate_batch(torch.from_numpy(blob).cuda(), d_out, items, block_type, chunk, flags, mode, d_dict,
                                  dicts)
        dev = d_out.cpu().numpy()
        assert int(rd["status"].max()) == 0
        written = np.zeros(total, dtype=bool)
        for o, m in zip(ooffs[:-1], rd["out_len"]):
            written[int(o):int(o) + int(m)] = True
        junk = rand_bytes(rng, blob.size, 256)
        for pinned in (True, False):
            if pinned:
                keep = torch.from_numpy(blob).pin_memory(), torch.empty(total, dtype=torch.uint8).pin_memory()
                h_in, h_out = keep[0].numpy(), keep[1].numpy()
            else:
                h_in, h_out = blob, np.empty(total, dtype=np.uint8)
            # a first call leaves other bytes in the library's staging buffers
            engine.deflate_batch_host(junk, h_out, items, block_type, chunk, flags, mode, h_dict, dicts)
            h_out[:] = SENTINEL
            rh = engine.deflate_batch_host(h_in, h_out, items, block_type, chunk, flags, mode, h_dict, dicts)
            for f in rd.dtype.names:
                assert np.array_equal(rh[f], rd[f]), (n, pinned, f)
            assert np.array_equal(h_out[written], dev[written]), (n, pinned)
            if n <= 600:  # (with more than 2048 copies the slack comes back zeroed)
                assert (h_out[~written] == SENTINEL).all(), (n, pinned)
