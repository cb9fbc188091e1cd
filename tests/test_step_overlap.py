"""The filter step's launch chain: tiles drawn from a queue in the call's scratch, kernels scheduled while the one
in front of them finishes.  Results must not depend on any of it.  Needs a GPU: -m gpu."""
import json

import numpy as np
import pytest

from conftest import alt_len_from_gfa_text, read_golden
from oracle import svjg_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from svjg import alnfilter, capi
    return alnfilter, capi, torch


def _tables(alnfilter, tag):
    edges = read_golden("c1_svs_edges.json" if tag == "c1" else f"{tag}_svs_edges.json.gz")
    return alnfilter.Tables.from_memory(edges, read_golden(f"{tag}.gfa.gz")).to_device(0)


def _hits(r):
    return sorted(zip(r.hit_sv2.tolist(), r.hit_off.tolist(), r.hit_len.tolist()))


def test_long_lines_at_the_head_pick_the_largest_tile(gpu):
    """The first 64 KiB, which size the tiles, hold lines of ~12 KB: the tile is the window's largest and most
    lines behind them fall into tiles of their own.  Counters and hits are those of the oracle and of a forced
    small tile."""
    alnfilter, capi, torch = gpu
    t = _tables(alnfilter, "c1")
    edges = json.loads(read_golden("c1_svs_edges.json"))
    alt = alt_len_from_gfa_text(read_golden("c1.gfa.gz"))
    base = read_golden("c1.gaf.gz").splitlines(True)
    lines = [l.rstrip("\n") + "\tcg:Z:" + "5M1I" * 3000 + "\n" for l in base[:8]] + base[8:]
    gaf = "".join(lines).encode()
    res = alnfilter.filter_host(t, gaf)
    want = O.hit_counts(O.filter_alignments(lines, edges, alt))
    got = {t.sv_ids[i]: [int(res.counts[i, 0]), int(res.counts[i, 1])] for i in range(t.num_sv) if res.counts[i].any()}
    assert got == {k: list(v) for k, v in want.items()}
    assert res.stats["n_records"] == len(lines)
    capi.check(capi.lib.svjg_filter_tune(capi.TUNE_TILE_BYTES, 1024))
    try:
        small = alnfilter.filter_host(t, gaf)
    finally:
        capi.check(capi.lib.svjg_filter_tune(capi.TUNE_TILE_BYTES, 0))
    assert (small.counts == res.counts).all() and _hits(small) == _hits(res)


@pytest.mark.parametrize("tag", ["s3", "s4"])
def test_back_to_back_calls_without_reset_accumulate(gpu, tag):
    """Three filter calls on one stream with no reset between them: every call zeroes its own tile queue and list
    cursors, so the counters and stats are exactly three times those of one call."""
    alnfilter, capi, torch = gpu
    t = _tables(alnfilter, tag)
    gaf = read_golden(f"{tag}.gaf.gz").encode()
    d = torch.frombuffer(bytearray(gaf), dtype=torch.uint8).cuda()
    one = alnfilter.DeviceFilter(t)
    one.reset()
    one.run(d)
    r1 = one.result()
    three = alnfilter.DeviceFilter(t, hit_cap=3 * r1.stats["n_hits"] + 8)
    three.reset()
    for _ in range(3):
        three.run(d)
    r3 = three.result()
    assert (r3.counts == 3 * r1.counts).all()
    for k in ("n_hits", "n_records", "n_multi", "n_checks", "n_exact"):
        assert r3.stats[k] == 3 * r1.stats[k], k
    assert _hits(r3) == sorted(_hits(r1) * 3)


def test_two_handles_on_two_streams_at_once(gpu):
    """Two filters with their own buffers run side by side on two streams (their scratch, tile queues included,
    is per call): each gives what it gives when the two run one after the other."""
    alnfilter, capi, torch = gpu
    tabs = [_tables(alnfilter, tag) for tag in ("s3", "s4")]
    data = [torch.frombuffer(bytearray(read_golden(f"{tag}.gaf.gz").encode()), dtype=torch.uint8).cuda() for tag in ("s3", "s4")]
    alone = []
    for t, d in zip(tabs, data):
        f = alnfilter.DeviceFilter(t)
        f.reset()
        f.run(d)
        alone.append(f.result())
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    filters = [alnfilter.DeviceFilter(t) for t in tabs]
    torch.cuda.synchronize()
    for _ in range(4):
        for f, d, s in zip(filters, data, streams):
            with torch.cuda.stream(s):
                f.reset()
                f.run(d)
    torch.cuda.synchronize()
    for f, want in zip(filters, alone):
        got = f.result()
        assert (got.counts == want.counts).all()
        assert got.stats == want.stats
        assert _hits(got) == _hits(want)
