"""Parity of the CUDA path (through the C ABI) against the golden outputs of the
unmodified reference and against the oracle.  Needs a GPU: -m gpu."""
import hashlib
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
    from svjg import alnfilter, capi, genotype
    return alnfilter, capi, genotype, torch


def _tables(alnfilter, tag):
    edges = read_golden("c1_svs_edges.json" if tag == "c1" else f"{tag}_svs_edges.json.gz")
    return alnfilter.Tables.from_memory(edges, read_golden(f"{tag}.gfa.gz")).to_device(0), edges


def _counts_dict(t, counts):
    return {t.sv_ids[i]: [int(counts[i, 0]), int(counts[i, 1])] for i in range(t.num_sv) if counts[i].any()}


@pytest.mark.parametrize("tag", ["c1", "s2", "s3", "s4"])
def test_filter_and_genotype_match_reference(gpu, tag, tmp_path):
    alnfilter, capi, genotype, torch = gpu
    t, edges = _tables(alnfilter, tag)
    gaf = read_golden(f"{tag}.gaf.gz").encode()
    res = alnfilter.filter_host(t, gaf)
    assert res.stats["n_records"] == gaf.count(b"\n")
    # JSON, byte for byte
    out = tmp_path / "x_informative_aln.json"
    alnfilter.write_informative_json(t, gaf, res, str(out))
    js = out.read_text()
    if tag == "c1":
        assert js == read_golden("c1_informative_aln.json.gz")
        want_counts = {k: [len(v[0]), len(v[1])] for k, v in json.loads(js).items()}
    else:
        assert hashlib.sha256(js.encode()).hexdigest() == read_golden(f"{tag}_informative_aln.sha256").strip()
        want_counts = json.loads(read_golden(f"{tag}_counts.json.gz"))
    assert _counts_dict(t, res.counts) == want_counts
    # genotype VCF, byte for byte
    vcf_lines = read_golden("c1.vcf" if tag == "c1" else f"{tag}.vcf.gz").splitlines(True)
    d_counts = torch.from_numpy(res.counts.view(np.int32)).cuda()
    text, n = genotype.genotype_vcf(t, d_counts, vcf_lines)
    assert text == read_golden("c1_genotype.vcf" if tag == "c1" else f"{tag}_genotype.vcf.gz")
    assert f"Genotyped svs: {n}\n" == read_golden(f"{tag}_stdout.txt")
    if tag == "c1":
        text2, _ = genotype.genotype_vcf(t, d_counts, vcf_lines, 40, 0.001)
        assert text2 == read_golden("c1_genotype_ms40_e1e-3.vcf")


def test_device_resident_path_equals_host_path(gpu):
    alnfilter, capi, genotype, torch = gpu
    t, _ = _tables(alnfilter, "s3")
    gaf = read_golden("s3.gaf.gz").encode()
    host = alnfilter.filter_host(t, gaf)
    d = torch.frombuffer(bytearray(gaf), dtype=torch.uint8).cuda()
    f = alnfilter.DeviceFilter(t, hit_cap=host.n_hits + 8)
    f.reset()
    f.run(d)
    r = f.result()
    assert (r.counts == host.counts).all()
    assert r.stats["n_hits"] == host.n_hits and r.stats["n_records"] == host.stats["n_records"]
    a = sorted(zip(r.hit_sv2.tolist(), r.hit_off.tolist(), r.hit_len.tolist()))
    b = sorted(zip(host.hit_sv2.tolist(), host.hit_off.tolist(), host.hit_len.tolist()))
    assert a == b
    # accumulate semantics: a second pass doubles the counters
    f.run(d)
    assert (f.counts.cpu().numpy().view(np.uint32) == 2 * host.counts).all()
    # more hits than the arrays hold: result() refuses to hand out a list cut short
    small = alnfilter.DeviceFilter(t, hit_cap=max(1, host.n_hits // 2))
    small.reset()
    small.run(d)
    with pytest.raises(capi.SvjgError) as exc:
        small.result()
    assert exc.value.code == capi.E_HITS_OVERFLOW
    assert (small.counts.cpu().numpy().view(np.uint32) == host.counts).all()


def test_quirk_cases(gpu, quirks, tmp_path):
    alnfilter, capi, genotype, torch = gpu
    t = alnfilter.Tables.from_memory(quirks["edges"], quirks["gfa"]).to_device(0)
    for case in quirks["cases"]:
        gaf = case["gaf"].encode()
        if case["rc"] == 0:
            res = alnfilter.filter_host(t, gaf)
            out = tmp_path / "q.json"
            alnfilter.write_informative_json(t, gaf, res, str(out))
            assert out.read_text() == case["json"], case["name"]
        else:
            with pytest.raises(alnfilter.InputError):
                alnfilter.filter_host(t, gaf)
                pytest.fail(case["name"])


def test_empty_and_tiny_inputs(gpu, tmp_path):
    alnfilter, capi, genotype, torch = gpu
    t, _ = _tables(alnfilter, "c1")
    res = alnfilter.filter_host(t, b"")
    assert res.n_hits == 0 and not res.counts.any()
    out = tmp_path / "e.json"
    alnfilter.write_informative_json(t, b"", res, str(out))
    assert out.read_text() == "{}"
    one = read_golden("c1.gaf.gz").splitlines(True)[0].encode()
    assert alnfilter.filter_host(t, one).stats["n_records"] == 1
    assert alnfilter.filter_host(t, one.rstrip(b"\n")).stats["n_records"] == 1


def test_tile_boundaries_and_long_lines(gpu):
    """Lines straddling 32 KiB tiles, lines longer than the look-ahead window
    (parsed from global memory) and read names padded so that line starts fall
    on every offset relative to the 16-byte scan chunks."""
    alnfilter, capi, genotype, torch = gpu
    t, edges = _tables(alnfilter, "c1")
    edges = json.loads(edges)
    alt = alt_len_from_gfa_text(read_golden("c1.gfa.gz"))
    base = read_golden("c1.gaf.gz").splitlines(True)[:400]
    lines = []
    for i, l in enumerate(base):
        cols = l.split("\t")
        cols[0] = cols[0] + "x" * (i % 37)
        l = "\t".join(cols)
        if i % 97 == 5:
            l = l.rstrip("\n") + "\tcg:Z:" + "5M1I" * 3000 + "\n"       # 12 KB > look-ahead
        if i % 131 == 7:
            l = l.rstrip("\n") + "\tzz:Z:" + "A" * 70000 + "\n"          # longer than a whole window
        lines.append(l)
    gaf = "".join(lines)
    res = alnfilter.filter_host(t, gaf.encode())
    want = O.hit_counts(O.filter_alignments(lines, edges, alt))
    assert _counts_dict(t, res.counts) == {k: list(v) for k, v in want.items()}
    assert res.stats["n_records"] == len(lines)


def test_genotype_kat40_and_random_vectors(gpu):
    alnfilter, capi, genotype, torch = gpu
    rows = [r.split("\t") for r in read_golden("kat40.tsv").splitlines()]
    cases = [(r[1], int(r[2]), int(r[3]), 3, 0.00005, r[4]) for r in rows]
    for row in read_golden("lik_random.tsv.gz").splitlines():
        ty, a, b, ms, e, geno, dp, numbers, prob = row.split("\t")
        cases.append((ty, int(a), int(b), int(ms), float(e), f"{geno}:{dp}:{numbers}:{prob}"))
    groups = {}
    for c in cases:
        groups.setdefault((c[3], c[4]), []).append(c)
    checked = 0
    for (ms, e), cs in groups.items():
        counts = torch.tensor([[c[1], c[2]] for c in cs], dtype=torch.int64).to(torch.int32).cuda()
        idx = np.arange(len(cs), dtype=np.uint32)
        ty = np.array([genotype.SVTYPE_CODE[c[0]] for c in cs], dtype=np.uint8)
        gt, flags, ad2, pl = genotype.genotype_device(counts, idx, ty, ms, e)
        for i, c in enumerate(cs):
            if c[1] == 0 and c[2] == 0:
                # a key with no hit never reaches likelihood() in the pipeline (gate :216)
                assert not flags[i] & capi.GT_GENOTYPED
                continue
            f = int(flags[i])
            h0, h1 = bool(f & capi.GT_HALVED_0), bool(f & capi.GT_HALVED_1)
            t1, t2 = int(ad2[i, 0]), int(ad2[i, 1])
            got = (f"{genotype.GT_TEXT[gt[i]]}:{genotype._num(t1 + t2, h0 or h1)}:"
                   f"{genotype._num(t1, h0)},{genotype._num(t2, h1)}:{pl[i, 0]},{pl[i, 1]},{pl[i, 2]}")
            assert got == c[5], c
            checked += 1
    assert checked > 27000


def test_genotype_oracle_sweep(gpu):
    """Dense sweep of small counts (every rounding / tie / min-support corner)
    against the oracle, all four SV types."""
    alnfilter, capi, genotype, torch = gpu
    pairs = [(a, b) for a in range(0, 41) for b in range(0, 41) if a or b]
    counts = torch.tensor(pairs, dtype=torch.int32).cuda()
    idx = np.arange(len(pairs), dtype=np.uint32)
    for name, code in genotype.SVTYPE_CODE.items():
        for ms in (0, 3, 7):
            gt, flags, ad2, pl = genotype.genotype_device(counts, idx, np.full(len(pairs), code, np.uint8), ms)
            for i, (a, b) in enumerate(pairs):
                g, dp, ad, p = O.genotype_counts(a, b, name, ms)
                assert genotype.GT_TEXT[gt[i]] == g and [str(x) for x in pl[i]] == p, (name, ms, a, b)


@pytest.mark.parametrize("tag", ["c1", "s2", "s3", "s4"])
def test_fast_path_equals_general_routine(gpu, tag):
    """The storage-free fast path and the quirk-exact general routine must give
    identical hits; the fast path must actually be taken for most lines."""
    alnfilter, capi, genotype, torch = gpu
    gaf = read_golden(f"{tag}.gaf.gz").encode()
    t_fast, _ = _tables(alnfilter, tag)
    t_gen, _ = _tables(alnfilter, tag)
    t_gen.set_flags(capi.FLAG_FORCE_GENERAL)
    a = alnfilter.filter_host(t_fast, gaf)
    b = alnfilter.filter_host(t_gen, gaf)
    assert (a.counts == b.counts).all()
    assert sorted(zip(a.hit_sv2.tolist(), a.hit_off.tolist())) == sorted(zip(b.hit_sv2.tolist(), b.hit_off.tolist()))
    assert b.stats["n_generic"] == b.stats["n_multi"] > 0
    assert a.stats["n_generic"] < 0.35 * a.stats["n_multi"], a.stats
    # exact-check mode probes more links but changes no result
    t_all, _ = _tables(alnfilter, tag)
    t_all.set_flags(capi.FLAG_EXACT_CHECKS)
    c = alnfilter.filter_host(t_all, gaf)
    assert (c.counts == a.counts).all() and c.stats["n_checks"] >= a.stats["n_checks"]
    assert c.stats["n_checks"] == b.stats["n_checks"]


def _oracle_counts(lines, edges_text, gfa_text):
    return O.hit_counts(O.filter_alignments(lines, json.loads(edges_text), alt_len_from_gfa_text(gfa_text)))


def _synthetic(name, scale, **kw):
    import io
    from svjg import synth
    g, vcf, gaf = synth.make_workload(name, scale=scale, **kw)
    buf = io.StringIO()
    g.write_gfa(buf)
    return g.edges_json(), buf.getvalue(), vcf, gaf


@pytest.mark.parametrize("name,scale", [("C2", 0.02), ("C3", 0.004), ("C4", 0.02), ("C5", 0.0002)])
def test_named_workloads_scaled_match_oracle(gpu, name, scale, tmp_path):
    """The BASELINE.json config shapes at a size the Python oracle finishes in seconds:
    counters, informative_aln.json (byte for byte) and the genotype VCF."""
    alnfilter, capi, genotype, torch = gpu
    edges_text, gfa_text, vcf, gaf = _synthetic(name, scale, cg_frac=0.05)
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    res = alnfilter.filter_host(t, gaf.encode())
    want = O.filter_alignments(gaf.splitlines(True), json.loads(edges_text), alt_len_from_gfa_text(gfa_text))
    assert _counts_dict(t, res.counts) == {k: list(v) for k, v in O.hit_counts(want).items()}
    out = tmp_path / "x.json"
    alnfilter.write_informative_json(t, gaf.encode(), res, str(out))
    assert out.read_text() == O.dumps_informative(want)
    d_counts = torch.from_numpy(res.counts.view(np.int32)).cuda()
    text, n = genotype.genotype_vcf(t, d_counts, vcf.splitlines(True))
    assert (text, n) == O.genotype_vcf(O.hit_counts(want), vcf.splitlines(True))
    assert res.stats["n_multi"] > 0 and res.n_hits > 0


def test_full_size_c2_properties(gpu):
    """BASELINE.json's C2 at full size (3 M records, ~0.5 GB): size-independent properties.
    Records seen = newlines; hits = sum of the counters; the chunked host path equals the
    single-shard device path; counters are additive over a cut at a line end; a slice of the
    batch matches the oracle exactly."""
    alnfilter, capi, genotype, torch = gpu
    edges_text, gfa_text, vcf, gaf = _synthetic("C2", 1.0)
    raw = gaf.encode()
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    host = alnfilter.filter_host(t, raw, want_hits=False)
    assert host.stats["n_records"] == raw.count(b"\n") == 3_000_000
    assert int(host.counts.sum()) == host.stats["n_hits"]
    d = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
    f = alnfilter.DeviceFilter(t, hit_cap=host.stats["n_hits"] + 8)
    f.reset()
    f.run(d)
    whole = f.result()
    assert (whole.counts == host.counts).all() and whole.stats["n_hits"] == host.stats["n_hits"]
    # every hit points at a whole line of the buffer
    off, ln = whole.hit_off.astype(np.int64), whole.hit_len.astype(np.int64)
    a = np.frombuffer(raw, dtype=np.uint8)
    assert (a[off + ln - 1] == 10).all() and ((off == 0) | (a[np.maximum(off, 1) - 1] == 10)).all()
    # additivity over a cut at a line end (what the multi-GPU sharding relies on)
    cut = raw.index(b"\n", len(raw) // 2) + 1
    left = alnfilter.filter_host(t, raw[:cut], want_hits=False)
    right = alnfilter.filter_host(t, raw[cut:], want_hits=False)
    assert (left.counts + right.counts == host.counts).all()
    # a slice against the oracle
    lines = gaf[:cut].splitlines(True)[:60000]
    part = alnfilter.filter_host(t, "".join(lines).encode(), want_hits=False)
    assert _counts_dict(t, part.counts) == {k: list(v) for k, v in _oracle_counts(lines, edges_text, gfa_text).items()}


def test_irregular_lines_take_the_exact_route(gpu):
    """CRLF line ends, read names longer than the fixed column spans, node names longer than the
    register path of the token kernel, 10-digit coordinates: all must equal the oracle."""
    alnfilter, capi, genotype, torch = gpu
    t, edges = _tables(alnfilter, "c1")
    edges = json.loads(edges)
    alt = alt_len_from_gfa_text(read_golden("c1.gfa.gz"))
    base = read_golden("c1.gaf.gz").splitlines(True)[:600]
    lines = []
    for i, l in enumerate(base):
        cols = l.rstrip("\n").split("\t")
        if i % 3 == 0:
            cols[0] = "Read_%d_length=8203bp_startpos=4333_number_of_errors=912_total_error_prob=0.1145_passes=1.9" % i
        if i % 5 == 0:
            cols[1] = cols[3] = "1234567890123"          # 13-digit Qlen / Qe: unused columns, any size is fine
        l = "\t".join(cols) + ("\r\n" if i % 4 == 1 else "\n")
        lines.append(l)
    gaf = "".join(lines)
    res = alnfilter.filter_host(t, gaf.encode())
    want = O.hit_counts(O.filter_alignments(lines, edges, alt))
    assert _counts_dict(t, res.counts) == {k: list(v) for k, v in want.items()}
    assert res.stats["n_records"] == len(lines) and res.stats["n_generic"] > 0
    # long node names and long coordinates in a private little graph
    long_chr = "a_very_long_contig_name_that_does_not_fit_in_thirty_two_bytes"
    n1, n2, n3 = f"{long_chr}:1-1000", f"{long_chr}:1001-2000", f"{long_chr}:4000000001-4000001000"
    edges2 = {f"{n1}@+@{n2}@+": [[f"{long_chr}:DEL-1000-1000", 0]], f"{n2}@+@{n3}@+": [[f"{long_chr}:DEL-2000-4000000000", 1]]}
    t2 = alnfilter.Tables.from_memory(json.dumps(edges2), "").to_device(0)
    rec = lambda path, tlen, ts, te: f"r\t3000\t0\t3000\t+\t{path}\t{tlen}\t{ts}\t{te}\t2900\t3000\t60\ttp:A:P\n"
    lines2 = [rec(f">{n1}>{n2}", 2000, 100, 1900), rec(f">{n1}>{n2}>{n3}", 3000, 100, 2900),
              rec(f"<{n2}<{n1}", 2000, 100, 1900), rec(f">{n2}>{n3}", 2000, 950, 1050)]
    res2 = alnfilter.filter_host(t2, "".join(lines2).encode())
    want2 = O.hit_counts(O.filter_alignments(lines2, edges2, {}))
    assert _counts_dict(t2, res2.counts) == {k: list(v) for k, v in want2.items()} and want2


def test_pool_exhaustion_falls_back_to_the_general_routine(gpu):
    """A line too long for the window is parsed where it lies with bitmaps from the exact kernel's bump
    pool (giant_line()); without room there, general() takes it: same counters and hits either way."""
    alnfilter, capi, genotype, torch = gpu
    step, n_nodes = 37, 700
    names = [f"chrL:{i * step + 1}-{(i + 1) * step}" for i in range(n_nodes)]
    edges = {f"{names[i]}@+@{names[i + 1]}@+": [[f"chrL:DEL-{(i + 1) * step}-{(i + 1) * step + 40}", 0]] for i in range(n_nodes - 1)}
    t = alnfilter.Tables.from_memory(json.dumps(edges), "").to_device(0)
    lines = []
    for k in (300, 450, 699):
        tlen = k * step
        path = "".join(">" + names[i] for i in range(k))
        lines.append(f"{'r' * 70}{k}\t{tlen}\t0\t{tlen}\t+\t{path}\t{tlen}\t150\t{tlen - 150}\t{tlen - 9}\t{tlen}\t60\ttp:A:P\n")
    gaf = "".join(lines).encode()
    normal = alnfilter.filter_host(t, gaf)
    capi.check(capi.lib.svjg_filter_tune(capi.TUNE_POOL_UNITS, 8))
    try:
        tiny = alnfilter.filter_host(t, gaf)
    finally:
        capi.check(capi.lib.svjg_filter_tune(capi.TUNE_POOL_UNITS, 0))
    want = O.hit_counts(O.filter_alignments(lines, edges, {}))
    assert want and _counts_dict(t, normal.counts) == {k: list(v) for k, v in want.items()}
    assert (tiny.counts == normal.counts).all() and tiny.n_hits == normal.n_hits
    assert normal.stats["n_generic"] == 0 and tiny.stats["n_generic"] == len(lines)
    assert sorted(zip(tiny.hit_sv2.tolist(), tiny.hit_off.tolist())) == sorted(zip(normal.hit_sv2.tolist(), normal.hit_off.tolist()))


def test_long_paths(gpu):
    """Paths of 2 .. 300 nodes on a private chain graph: up to 32 nodes go through the ordinary rounds,
    longer ones (up to 256) through long_line() -- all equal to the oracle and not generic.  A path that
    revisits a node follows the first-occurrence rules: in place in an ordinary round, on the exact route
    where the path is longer than a round."""
    alnfilter, capi, genotype, torch = gpu
    n_nodes, step = 330, 37
    names = [f"chrL:{i * step + 1}-{(i + 1) * step}" for i in range(n_nodes)]
    edges = {}
    for i in range(n_nodes - 1):
        edges[f"{names[i]}@+@{names[i + 1]}@+"] = [[f"chrL:DEL-{(i + 1) * step}-{(i + 1) * step + 40}", 0]]
    for i in range(0, n_nodes - 2, 7):                                   # deletions that jump over one node
        edges[f"{names[i]}@+@{names[i + 2]}@+"] = [[f"chrL:DEL-{(i + 1) * step}-{(i + 2) * step}", 1]]
    t = alnfilter.Tables.from_memory(json.dumps(edges), "").to_device(0)

    def rec(idx, ts, te, fwd=True):
        tlen = len(idx) * step
        path = "".join(">" + names[i] for i in idx) if fwd else "".join("<" + names[i] for i in reversed(idx))
        return f"read\t{tlen}\t0\t{tlen}\t+\t{path}\t{tlen}\t{ts}\t{te}\t{tlen - 9}\t{tlen}\t60\ttp:A:P\tcm:i:7\n"

    lines, n_over = [], 0
    for k in (2, 3, 17, 31, 32, 33, 34, 40, 47, 63, 64, 65, 70, 96, 97, 128, 200, 256, 257, 300):
        for start in (0, 5, 14):
            idx = list(range(start, start + k))
            if k % 2 == 1 and start == 0:
                idx = [0, 2] + list(range(3, k + 1))                     # uses a jump link
            tlen = len(idx) * step
            for ts, te in ((tlen // 5, tlen - tlen // 4), (3, tlen - 2), (0, tlen - 1)):
                lines += [rec(idx, ts, te, True), rec(idx, ts, te, False)]
                n_over += 2 * (len(idx) > 256)                           # more nodes than long_line() keeps: exact route
    res = alnfilter.filter_host(t, "".join(lines).encode())
    want = O.hit_counts(O.filter_alignments(lines, edges, {}))
    assert want and _counts_dict(t, res.counts) == {k: list(v) for k, v in want.items()}
    # more than 256 nodes, or longer than the look-ahead (1 KiB) and straddling a tile end: the exact
    # kernel takes the line, but its giant_line() applies the fast rules there -- still not generic
    assert res.stats["n_multi"] == len(lines) and res.stats["n_generic"] == 0 and n_over > 0
    # revisits: node 10 comes twice (first-occurrence rules), once in a short and once in a long path
    loops = [rec(list(range(0, 20)) + [10, 11, 12], 120, 700), rec(list(range(0, 50)) + [10, 11], 120, 1700),
             rec(list(range(60, 0, -1)), 100, 2000), rec([0] + list(range(44, 1, -1)) + [45, 46], 20, 1600)]
    res2 = alnfilter.filter_host(t, "".join(loops).encode())
    want2 = O.hit_counts(O.filter_alignments(loops, edges, {}))
    assert _counts_dict(t, res2.counts) == {k: list(v) for k, v in want2.items()}
    # the short revisit is resolved in the ordinary round (the first twin's lane has the first-occurrence strand and
    # the first-index sums), the long one takes the exact route; an inverted stretch is no revisit
    assert res2.stats["n_generic"] == 1 and res2.stats["n_multi"] == 4


def test_paths_that_revisit_nodes(gpu):
    """conftest.revisit_walks: names that come twice in a path (loops, `>A>A`, `>A<A`) are resolved in the ordinary
    rounds from the lane of their first occurrence -- counters and the stored lines equal the oracle's, and no
    such line needs the general routine; with the general routine forced the result is the same."""
    from conftest import revisit_walks
    alnfilter, capi, genotype, torch = gpu
    edges, lines = revisit_walks()
    gaf = "".join(lines).encode()
    want = O.filter_alignments(lines, edges, {})
    t = alnfilter.Tables.from_memory(json.dumps(edges), "").to_device(0)
    res = alnfilter.filter_host(t, gaf)
    assert _counts_dict(t, res.counts) == {k: list(v) for k, v in O.hit_counts(want).items()}
    got = {}
    order = np.lexsort((res.hit_sv2, res.hit_off))
    for s2, o, n in zip(res.hit_sv2[order].tolist(), res.hit_off[order].tolist(), res.hit_len[order].tolist()):
        got.setdefault(t.sv_ids[s2 >> 1], [[], []])[s2 & 1].append(O.kept_text(gaf[o:o + n].decode()))
    assert {k: [sorted(v[0]), sorted(v[1])] for k, v in got.items()} == {k: [sorted(v[0]), sorted(v[1])] for k, v in want.items()}
    assert res.stats["n_generic"] == 0 and res.stats["n_multi"] == len(lines)
    t.set_flags(capi.FLAG_FORCE_GENERAL)
    gen = alnfilter.filter_host(t, gaf)
    assert (gen.counts == res.counts).all() and gen.stats["n_generic"] == gen.stats["n_multi"] == len(lines)


@pytest.mark.parametrize("tile", [1024, 1600, 3072, 3360, 4992])
def test_every_tile_size_gives_the_same_result(gpu, tile):
    """The probe kernel picks the bytes per tile from the line length; any tile size must give the
    same counters and hits (SVJG_TUNE_TILE_BYTES forces one)."""
    alnfilter, capi, genotype, torch = gpu
    t, _ = _tables(alnfilter, "s3")
    gaf = read_golden("s3.gaf.gz").encode()
    normal = alnfilter.filter_host(t, gaf)
    capi.check(capi.lib.svjg_filter_tune(capi.TUNE_TILE_BYTES, tile))
    try:
        forced = alnfilter.filter_host(t, gaf)
    finally:
        capi.check(capi.lib.svjg_filter_tune(capi.TUNE_TILE_BYTES, 0))
    same = lambda st: {k: v for k, v in st.items() if k != "n_exact"}     # lines past the window depend on the tile
    assert (forced.counts == normal.counts).all() and same(forced.stats) == same(normal.stats)
    assert sorted(zip(forced.hit_sv2.tolist(), forced.hit_off.tolist())) == sorted(zip(normal.hit_sv2.tolist(), normal.hit_off.tolist()))


def test_host_buffers_and_torch_free_paths(gpu, tmp_path):
    """Page-locked inputs and outputs (PinnedBytes, RegisteredBytes, HostBuffers: the kernels write the hits
    straight into them) and svjg_genotype_host give what the pageable / tensor paths give."""
    alnfilter, capi, genotype, torch = gpu
    t, _ = _tables(alnfilter, "s3")
    raw = read_golden("s3.gaf.gz").encode()
    want = alnfilter.filter_host(t, raw)                               # pageable in, pageable out
    key = lambda r: sorted(zip(r.hit_sv2.tolist(), r.hit_off.tolist(), r.hit_len.tolist()))
    p = tmp_path / "s3.gaf"
    p.write_bytes(raw)
    pinned = alnfilter.read_file_pinned(str(p))
    assert bytes(pinned.array) == raw
    reg = alnfilter.RegisteredBytes(np.frombuffer(bytearray(raw), dtype=np.uint8))
    out = alnfilter.HostBuffers(t, want.n_hits + 5)
    for src in (pinned, reg):
        got = alnfilter.filter_host(t, src, out=out)
        assert (got.counts == want.counts).all() and got.stats == want.stats and key(got) == key(want)
    with pytest.raises(RuntimeError):
        alnfilter.filter_host(t, pinned, out=alnfilter.HostBuffers(t, 3))
    # genotype from host arrays == genotype from device tensors
    header, recs = genotype.parse_vcf(read_golden("s3.vcf.gz").splitlines(True))
    idx = np.array([capi.NO_SV if (r[2] is None or t.find_sv(r[2]) is None) else t.find_sv(r[2]) for r in recs], dtype=np.uint32)
    ty = np.array([r[1] for r in recs], dtype=np.uint8)
    a = genotype.genotype_host(want.counts, idx, ty)
    d_counts = torch.from_numpy(want.counts.view(np.int32)).cuda()
    b = genotype.genotype_device(d_counts, idx, ty)
    c = genotype.genotype_device(d_counts, torch.from_numpy(idx.view(np.int32)).cuda(), torch.from_numpy(ty).cuda())
    for x, y, z in zip(a, b, c):
        assert (x == y).all() and (x == z).all()
    text_host, n_host = genotype.genotype_vcf(t, want.counts, read_golden("s3.vcf.gz").splitlines(True))
    assert text_host == read_golden("s3_genotype.vcf.gz")


def test_damaged_lines_match_the_reference(gpu, tmp_path):
    """tests/golden/fuzz_lines.json.gz: 2500 randomly damaged GAF lines, each run alone as a file through
    the UNMODIFIED reference (tests/golden/make_fuzz.py).  Where it exits with status 1 the CUDA path
    must report an input error, elsewhere the counters must be equal.  Like the command-line front-end,
    the bytes first get the reference's text-mode line ends (a carriage return ends a line)."""
    alnfilter, capi, genotype, torch = gpu
    t, _ = _tables(alnfilter, "c1")
    fx = json.loads(read_golden("fuzz_lines.json.gz"))
    n_err = n_hit = 0
    for c in fx["cases"]:
        raw = alnfilter.translate_newlines(c["line"].encode("utf-8"))
        try:
            res = alnfilter.filter_host(t, raw, want_hits=False)
            got = _counts_dict(t, res.counts)
            failed = False
        except alnfilter.InputError:
            failed = True
        assert failed == bool(c["rc"]), c["line"]
        if not failed:
            assert got == c["counts"], c["line"]
            n_hit += bool(got)
        n_err += failed
    assert n_err > 500 and n_hit > 500
    # a whole file with CR LF line ends: the JSON stores "\n", byte for byte as the reference writes it
    raw = alnfilter.translate_newlines(fx["crlf"]["gaf"].encode())
    res = alnfilter.filter_host(t, raw)
    out = tmp_path / "crlf.json"
    alnfilter.write_informative_json(t, raw, res, str(out))
    assert out.read_text() == fx["crlf"]["json"]


def test_damaged_vcfs_match_the_reference(gpu):
    """tests/golden/fuzz_vcf.json.gz: 800 small VCFs with one damaged body line, run through the UNMODIFIED
    predict-genotype.py.  The host mirror + genotype kernel must fail where it exits with status 1 and
    write the same text and count elsewhere."""
    import io
    alnfilter, capi, genotype, torch = gpu
    counts = genotype.AlnCounts.from_memory(read_golden("c1_informative_aln.json.gz"))
    cases = json.loads(read_golden("fuzz_vcf.json.gz"))
    n_err = 0
    for c in cases:
        lines = list(io.StringIO(c["vcf"], newline=None))                 # text mode, like open()
        try:
            text, n = genotype.genotype_vcf_from_json(counts, lines, c["ms"], 0.00005)
            failed = False
        except (genotype.VcfError, capi.SvjgError, ValueError):
            failed = True
        assert failed == bool(c["rc"]), c["vcf"][-400:]
        if not failed:
            assert text == c["out"], c["vcf"][-400:]
            assert f"Genotyped svs: {n}\n" == c["stdout"]
        n_err += failed
    assert n_err > 100


def test_damaged_link_tables_match_the_reference(gpu, tmp_path):
    """tests/golden/fuzz_edges.json: 300 svs_edges.json variants with damaged entries, each run through the
    UNMODIFIED reference filter on 150 c1 lines (tests/golden/make_fuzz.py regenerates the variants from
    its seed): same exit status, same informative_aln.json bytes."""
    import hashlib
    import importlib.util
    import os
    alnfilter, capi, genotype, torch = gpu
    spec = importlib.util.spec_from_file_location("make_fuzz", os.path.join(os.path.dirname(__file__), "golden", "make_fuzz.py"))
    mf = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mf)
    gfa = read_golden("c1.gfa.gz")
    raw = "".join(mf.edges_gaf_lines()).encode()
    want = json.loads(read_golden("fuzz_edges.json"))
    out = tmp_path / "x.json"
    for text, c in zip(mf.damaged_edges(len(want)), want):
        t = alnfilter.Tables.from_memory(text, gfa).to_device(0)
        try:
            res = alnfilter.filter_host(t, raw)
            alnfilter.write_informative_json(t, raw, res, str(out))
            got = (0, hashlib.sha256(out.read_bytes()).hexdigest())
        except alnfilter.InputError:
            got = (1, None)
        assert got[0] == c["rc"]
        if not got[0]:
            assert got[1] == c["sha256"]
        t.close()
