"""The scan kernel's fast route at the edges of what it accepts, against the oracles.

A seeded generator in this file writes GAF lines on a private graph, in families that are batches of their own:
A node names (chroms of 1 to 17 bytes, every alignment of a name start, 1- to 10-digit coordinates, `.k` alt
nodes, second colons, leading zeros), B column widths around the 32- and 64-bit windows of the line-shape test,
C overlap margins equal to d_over and d_over - 1, D the packing of path nodes into rounds of 32 lanes, and
E all of them shuffled with C2-style lines and the damaged lines of fuzz_lines.json.gz that the reference
accepts.  The CPU part holds the two oracles against each other on these batches and the two node tables of
the library against each other on every generated name; the GPU part holds the CUDA path against the C oracle:
counters, hit tuples, the route each batch takes, and on E the device-rendered JSON, the resident route and
every launch-geometry knob."""
import io
import json
import random
import string

import numpy as np
import pytest

from conftest import alt_len_from_gfa_text, read_golden
from oracle import svjg_oracle as O

SEED = 20261021
ALPHABET = string.ascii_letters + string.digits + "_.-*"

# batches whose lines are all plain by the rules of DESIGN.md section 4: every line stays on the fast route
PLAIN = ("A_plain", "B_plain", "C_d0", "C_d1", "C_d100", "C_d1e9", "A_utf8")
# every line irregular: each one goes to the exact kernel; the node kinds (a name the fast route cannot key)
# also end in the general routine
IRREGULAR_NODES = ("A_chrom16", "A_colon2", "A_digits10", "A_zero", "A_v1_lt_v0", "A_alt_absent", "A_alt_len0")
IRREGULAR_LINES = ("B_irregular",)
OTHER = ("B_wide", "B_no_final_newline", "D_rounds", "E")
D_OVER = {"C_d0": 0, "C_d1": 1, "C_d100": 100, "C_d1e9": 10 ** 9}
ASCII_BATCHES = tuple(n for n in PLAIN + IRREGULAR_NODES + IRREGULAR_LINES + OTHER if n != "A_utf8")


class Graph:
    """A private graph: link keys with one entry each, alt-node lengths (the GFA's S lines)."""

    def __init__(self):
        self.edges = {}
        self.alt = {}
        self.gfa = []

    def link(self, a, b):
        key = f"{a}@+@{b}@+"
        assert key not in self.edges, key
        n = len(self.edges)
        self.edges[key] = [[f"E{n // 2}:sv", n % 2]]

    def chain(self, names):
        for a, b in zip(names, names[1:]):
            self.link(a, b)

    def alt_node(self, name, length):
        """length None: the node has no S line; 0: an S line with an empty sequence."""
        if length is None:
            return
        self.alt[name] = length
        self.gfa.append(f"S\t{name}\t{'ACGT' * (length // 4) + 'ACG'[:length % 4]}\tLN:i:{length}\n")

    def node_len(self, name):
        last = name.rsplit(":", 1)[1]
        if "." in last:
            return self.alt.get(name, 0)
        v0, v1 = last.split("-")
        return int(v1) - int(v0) + 1

    @property
    def gfa_text(self):
        return "".join(self.gfa)


def gaf_line(qname, path, tlen, ts, te, cols24=("1000", "0", "1000"), strand="+", nm="900", alen="1000", mapq="60",
             tags="\ttp:A:P\tcm:i:7", end="\n"):
    return "\t".join([qname, *cols24, strand, path, str(tlen), str(ts), str(te), nm, alen, mapq]) + tags + end


def path_of(names, fwd=True):
    return "".join(">" + n for n in names) if fwd else "".join("<" + n for n in reversed(names))


def path_lens(g, names, fwd=True):
    order = names if fwd else list(reversed(names))
    return [g.node_len(n) for n in order]


class Batch:
    def __init__(self, name, d_over=100):
        self.name, self.d_over, self.lines, self.size = name, d_over, [], 0

    def add(self, line):
        self.lines.append(line)
        self.size += len(line.encode())

    def add_aligned(self, make, align):
        """make(qname) -> line; the read name is padded so that the path's first name starts at a byte offset
        that is `align` modulo 4 (the tiles are multiples of 32 bytes: the offset in the window has the same
        alignment)."""
        q = f"q{len(self.lines)}"
        line = make(q)
        head = len("\t".join(line.split("\t")[:5]).encode()) + 2          # tab and the first '>' or '<'
        pad = (align - (self.size + head)) % 4
        self.add(make(q + "x" * pad))

    @property
    def raw(self):
        return "".join(self.lines).encode()


def name_spans(lines):
    """(byte offset, name) of every path name in the concatenated lines."""
    out, off = [], 0
    for line in lines:
        b = line.encode()
        cols = b.split(b"\t")
        if len(cols) > 5 and cols[5][:1] in (b">", b"<"):
            p = off + len(b"\t".join(cols[:5])) + 1
            path = cols[5]
            i = 0
            while i < len(path):
                j = i + 1
                while j < len(path) and path[j:j + 1] not in (b">", b"<"):
                    j += 1
                out.append((p + i + 1, path[i + 1:j].decode()))
                i = j
        off += len(b)
    return out


def _chroms(rng):
    out = []
    for n in range(1, 18):
        for _ in range(3):
            c = "".join(rng.choice(ALPHABET) for _ in range(n))
            if c not in out:
                out.append(c)
    # real reference names (16 and more bytes are declined by both key builders), prefixes of each other,
    # and names that differ only in byte 14 (the last chrom byte in front of the length byte)
    out += ["chrEBV", "KI270728.1", "NC_000001.11", "chr22_KI270731v1_random", "chrUn_KI270742v1",
            "chr1", "chr1_", "chr10", "chr5_GL000208v1", "chr5_GL000208v2", "NT_187361.1abcd", "NT_187361.1abce"]
    return list(dict.fromkeys(out))


def _coords(rng):
    """(start, end) pairs of one chain: starts and ends of 1 to 9 digits, a 0 start, 1-bp nodes; all starts distinct."""
    while True:
        specs = [(0, 9), (2, 7), (1, 1)]
        for d in range(1, 10):
            v0 = rng.randrange(3, 10) if d == 1 else rng.randrange(10 ** (d - 1), 10 ** d)
            v1 = min(v0 + rng.randrange(20, 400), 10 ** 9 - 1)
            specs.append((v0, v1))
        v = rng.randrange(100000, 999999)
        specs.append((v, v))                                               # a 1-bp node
        specs.append((999999000 + rng.randrange(0, 99), 999999999))        # a 9-digit end
        if len({s for s, _ in specs}) == len(specs):
            return specs


def _chain_names(rng, chrom):
    specs = _coords(rng)
    names = [f"{chrom}:{a}-{b}" for a, b in specs]
    alt = f"{chrom}:{specs[3][1] + 1}.1"                                   # an alt node behind a ref node
    rng.shuffle(names)
    names.insert(len(names) // 2, alt)
    return names, alt


def _margins(lens, rng):
    tlen = max(1, sum(max(x, 0) for x in lens))
    ts = rng.randrange(0, max(1, lens[0] // 3 + 1))
    te = max(ts, tlen - 1 - rng.randrange(0, max(1, lens[-1] // 3 + 1)))
    return tlen, ts, te


def family_a(g, rng, batches):
    """Node names.  A_plain: every chrom of at most 15 bytes, every alignment, both orientations."""
    chroms = _chroms(rng)
    plain = batches["A_plain"]
    for chrom in chroms:
        names, alt = _chain_names(rng, chrom)
        g.chain(names)
        g.alt_node(alt, rng.randrange(1, 60))
        target = plain if len(chrom.encode()) <= 15 else batches["A_chrom16"]
        for align in range(4):
            for fwd in (True, False):
                k = len(names) if fwd == (align % 2 == 0) else rng.randrange(2, len(names))
                s = rng.randrange(0, len(names) - k + 1)
                sub = names[s:s + k]
                lens = path_lens(g, sub, fwd)
                tlen, ts, te = _margins(lens, rng)
                target.add_aligned(lambda q: gaf_line(q, path_of(sub, fwd), tlen, ts, te), align)

    def irregular(batch, chrom, bad, length=None, linked=True):
        """A chain on `chrom` with the node `bad` in its middle."""
        names = [f"{chrom}:{10001 + 300 * k}-{10300 + 300 * k}" for k in range(6)]
        names.insert(3, bad)
        if linked:
            g.chain(names)
        g.alt_node(bad, length)
        for align in range(4):
            for fwd in (True, False):
                sub = names if linked else names[2:4]
                lens = path_lens(g, sub, fwd)
                tlen, ts, te = _margins(lens, rng)
                batch.add_aligned(lambda q: gaf_line(q, path_of(sub, fwd), tlen, ts, te), align)

    for i, chrom in enumerate(["HLA-A*01:01", "a:b", ":", "chr1:x"]):                # a second colon
        irregular(batches["A_colon2"], chrom + "x" * i, f"{chrom}:{1000 + i}-{2000 + i}")
    for i in range(4):                                                                 # 10-digit start / end
        irregular(batches["A_digits10"], f"dten{i}", f"dten{i}:{1234567890 + i}-{1234568890 + i}")
        irregular(batches["A_digits10"], f"dtn{i}", f"dtn{i}:{999999900 + i}-{1000000100 + i}")
    for i in range(4):                                                                 # leading zeros
        irregular(batches["A_zero"], f"zero{i}", f"zero{i}:0{300 + i}-{900 + i}")
        irregular(batches["A_zero"], f"zro{i}", f"zro{i}:{300 + i}-0{900 + i}")
    for i in range(4):
        irregular(batches["A_v1_lt_v0"], f"down{i}", f"down{i}:{5000 + i}-{4990 + i}")
        # an alt node without an S line: only in a line with no link (the reference raises on its length otherwise)
        irregular(batches["A_alt_absent"], f"noalt{i}", f"noalt{i}:{7000 + i}.1", None, linked=False)
        irregular(batches["A_alt_len0"], f"zalt{i}", f"zalt{i}:{7000 + i}.1", 0)
    return chroms


def _int_text(n, first="1"):
    """n digits, not starting with '0'."""
    return (first + "234567890" * 3)[:n]


def _cols_for_run(run, tlen, ts, te, tags):
    """Nmatch, Alen and Mapq so that columns 7-12 with their tabs take `run` bytes."""
    rest = run - len(str(tlen)) - len(str(ts)) - len(str(te)) - (6 if tags else 5)
    nm = min(18, rest - 2)
    alen = min(18, rest - nm - 1)
    mapq = rest - nm - alen
    assert 1 <= mapq <= 18 and nm >= 1 and alen >= 1
    return _int_text(nm, "9"), _int_text(alen, "9"), _int_text(mapq, "6")


def family_b(g, rng, batches):
    """Column widths.  Three 1 kb nodes, and three nodes of 300 Mb for 9- and 10-digit Tlen, Ts and Te."""
    names = [f"colB:{1000 * i + 1}-{1000 * (i + 1)}" for i in range(4)]
    g.chain(names)
    big = [f"colBig:{300000000 * i + 1}-{300000000 * (i + 1)}" for i in range(3)]
    g.chain(big)
    p3, tl = path_of(names[:3]), 3000
    pl, wide, irr = batches["B_plain"], batches["B_wide"], batches["B_irregular"]
    for n in (1, 31, 32, 33, 63, 64, 65, 200):                                  # read names
        q = ("R" + "n" * n)[:n]
        for fwd in (True, False):
            pl.add(gaf_line(q, path_of(names[:3], fwd), tl, 150, 2800))
    for run in (30, 31, 32, 33, 34):                                            # columns 2-4 and their tabs
        d = run - 3
        cols = (_int_text(d - 2 * (d // 3)), _int_text(d // 3), _int_text(d // 3))
        for strand in ("+", "-"):
            (pl if run <= 31 else wide).add(gaf_line(f"c24_{run}", p3, tl, 120, 2850, cols24=cols, strand=strand))
    for tags in ("\ttp:A:P", ""):                                               # columns 7-12 and their tabs
        for run in (62, 63, 64, 65, 66):
            nm, alen, mapq = _cols_for_run(run, tl, 130, 2870, tags)
            line = gaf_line(f"c712_{run}", p3, tl, 130, 2870, nm=nm, alen=alen, mapq=mapq, tags=tags)
            (pl if run <= 63 else wide).add(line)
    # Ts = 0, Te = Tlen - 1 (tail 0), Te = Tlen (tail -1), Ts > Te, margins right at d_over
    for ts, te in ((0, tl - 1), (0, tl), (900, 2999), (1900, 1100), (900, 2100), (899, 2101), (901, 2099)):
        for fwd in (True, False):
            pl.add(gaf_line("edge", path_of(names[:3], fwd), tl, ts, te))
    pl.add(gaf_line("ts_zeros", p3, tl, "000000150", "000002800"))              # 9 digits with leading zeros
    pl.add(gaf_line("strand2", p3, tl, 150, 2800, strand="+-"))                 # a two-byte strand column
    pl.add(gaf_line("notags", p3, tl, 150, 2800, tags=""))
    # 9 digits in Tlen, Ts and Te: the fast route; 10 digits: the exact route
    pb = path_of(big)
    for tlen, ts, te in ((900000000, 123456789, 876543210), (999999999, 299999899, 699999999),
                         (900000000, 300000000 - 100, 600000000 + 99)):
        pl.add(gaf_line("big9", pb, tlen, ts, te))
        pl.add(gaf_line("big9r", path_of(big, False), tlen, ts, te))
    for tlen, ts, te in ((1000000000, 123456789, 876543210), (900000000, "0123456789", 876543210),
                         (1500000000, 100, 1000000000)):
        irr.add(gaf_line("big10", pb, tlen, ts, te))
    irr.add(gaf_line("alen0", p3, tl, 150, 2800, alen="0999"))                  # Alen with a leading 0
    irr.add(gaf_line("alen0", p3, tl, 150, 2800, nm="0", alen="01000", tags=""))
    pl.add(gaf_line("last", p3, tl, 150, 2800, tags=""))                        # twelve columns at the end of the file
    nofinal = batches["B_no_final_newline"]
    for line in pl.lines[:-1]:
        nofinal.add(line)
    nofinal.add(pl.lines[-1].rstrip("\n"))


def family_c(g, rng, batches):
    """Overlap margins: every link of every line is placed once with its left and its right margin equal to
    d_over and d_over - 1 (the other margin as it falls)."""
    small = [f"ovl:{100 * i + 1}-{100 * i + 50 + 13 * i}" for i in range(5)]
    g.chain(small)
    huge = [f"ovlh:{i + 1}-{600000000 + i}" for i in range(4)]                  # 6e8 bases each: margins of 1e9
    g.chain(huge)
    for bname, dov in D_OVER.items():
        b = batches[bname]
        b.d_over = dov
        for names in (small, huge):
            for fwd in (True, False):
                lens = path_lens(g, names, fwd)
                for i in range(1, len(names)):
                    left_sum, right_sum = sum(lens[:i]), sum(lens[i:])
                    for ml in (dov, dov - 1):
                        for mr in (dov, dov - 1):
                            ts, tail = left_sum - ml, right_sum - mr
                            tlen = max(999999999 if names is huge else 5000, tail + 1)
                            te = tlen - 1 - tail
                            if ts < 0 or te < 0 or max(tlen, ts, te) >= 10 ** 9:
                                continue
                            b.add(gaf_line(f"m{ml - dov}{mr - dov}", path_of(names, fwd), tlen, ts, te))
        assert len(b.lines) >= 8, bname


def family_d(g, rng, batches, irregular_lines):
    """Round packing: node counts that fill a round of 32 lanes exactly or overflow it by one, name twins on
    lanes 0 and 31, one-node and irregular lines in between."""
    names = [f"rnd:{50 * i + 1}-{50 * (i + 1)}" for i in range(80)]
    g.chain(names)
    b = batches["D_rounds"]
    n_irr = 0

    def multi(k, s=None, fwd=True):
        s = rng.randrange(0, len(names) - k + 1) if s is None else s
        sub = names[s:s + k]
        tlen = 50 * k
        b.add(gaf_line(f"k{k}", path_of(sub, fwd), tlen, 20, tlen - 20))

    def one():
        b.add(gaf_line("one", ">" + names[rng.randrange(80)], 50, 5, 45))

    def irr():
        nonlocal n_irr
        b.add(rng.choice(irregular_lines))
        n_irr += 1

    groups = [[32], [31, 2], [30, 2], [16, 16], [32, 33], [33], [2] * 16, [4] * 8, [8] * 4, [3] * 10 + [2],
              [31], [1, 31], [17, 15], [15, 17], [33, 32]]
    for rep in range(3):
        for grp in groups:
            for k in grp:
                multi(k, fwd=rng.random() < 0.7) if k > 1 else one()
                if rep == 1:
                    one()
                if rep == 2 and rng.random() < 0.3:
                    irr()
        # a full round, then a line whose name comes again on lane 31 (the same strand, then the other one)
        multi(32)
        tw = names[10:41] + [names[10]]
        b.add(gaf_line("twin", path_of(tw), 1600, 20, 1580))
        multi(32)
        b.add(gaf_line("twin2", path_of(names[10:41]) + "<" + names[10], 1600, 20, 1580))
        irr()
    return n_irr


def _fuzz_lines():
    fx = json.loads(read_golden("fuzz_lines.json.gz"))
    out = []
    for c in fx["cases"]:
        line = c["line"]
        if c["rc"] or "\r" in line or not line.isascii():
            continue
        out.append(line if line.endswith("\n") else line + "\n")
    return out


def _synth_c2(scale=0.004):
    from svjg import synth
    g, _vcf, gaf = synth.make_workload("C2", scale=scale)
    buf = io.StringIO()
    g.write_gfa(buf)
    return json.loads(g.edges_json()), buf.getvalue(), gaf.splitlines(True)


def utf8_batch(rng):
    """Chroms whose bytes are not all ASCII, the last byte of the chrom included (UTF-8 continuation bytes have
    bit 7 set): in a chrom of 13 to 15 bytes that byte lies in the fourth key word."""
    g = Graph()
    b = Batch("A_utf8")
    chroms = []
    for n in range(2, 16):
        chroms.append("".join(rng.choice(string.ascii_letters) for _ in range(n - 2)) + "é")
    chroms += ["chrÜ", "Ωmega_contig12", "contig_ßß_α", "xxxxxxxxxxxx→"]
    for chrom in chroms:
        assert len(chrom.encode()) <= 15
        names, alt = _chain_names(rng, chrom)
        g.chain(names)
        g.alt_node(alt, rng.randrange(1, 60))
        for align in range(4):
            fwd = align % 2 == 0
            lens = path_lens(g, names, fwd)
            tlen, ts, te = _margins(lens, rng)
            b.add_aligned(lambda q: gaf_line(q, path_of(names, fwd), tlen, ts, te), align)
    return g, b, chroms


def generate(seed=SEED, with_e=True):
    """{batch name: Batch}, the private graph, and for E its merged tables (edges dict, GFA text)."""
    rng = random.Random(seed)
    g = Graph()
    names = PLAIN + IRREGULAR_NODES + IRREGULAR_LINES + OTHER
    batches = {n: Batch(n) for n in names if n not in ("A_utf8",)}
    chroms = family_a(g, rng, batches)
    family_b(g, rng, batches)
    family_c(g, rng, batches)
    irregular_lines = [l for n in IRREGULAR_NODES for l in batches[n].lines if n != "A_alt_absent"]
    n_irr_d = family_d(g, rng, batches, irregular_lines)
    ug, ub, uchroms = utf8_batch(rng)
    out = {"batches": batches, "graph": g, "chroms": chroms, "n_irr_d": n_irr_d, "utf8": (ug, ub, uchroms)}
    if with_e:
        edges, gfa, c2 = _synth_c2()
        c1_edges = json.loads(read_golden("c1_svs_edges.json"))
        for other in (edges, c1_edges):
            assert not set(other) & set(g.edges)
        merged = {**c1_edges, **edges, **g.edges}
        assert len(merged) == len(c1_edges) + len(edges) + len(g.edges)
        alt_merged = {**alt_len_from_gfa_text(read_golden("c1.gfa.gz")), **alt_len_from_gfa_text(gfa)}
        assert not set(alt_merged) & set(g.alt)
        gfa_text = read_golden("c1.gfa.gz") + gfa + g.gfa_text
        pool = [l for n in ASCII_BATCHES if n not in ("B_no_final_newline", "E") for l in batches[n].lines]
        pool += c2 + _fuzz_lines()
        last = batches["B_plain"].lines[-1].rstrip("\n")                        # twelve columns, no newline
        rng.shuffle(pool)
        for line in pool:
            batches["E"].add(line)
        batches["E"].add(last)
        out["e_tables"] = (merged, gfa_text)
    else:
        del batches["E"]
    return out


def tables_for(gen, name):
    """(edges dict, GFA text, alt-length dict) the batch runs against."""
    if name == "E":
        edges, gfa = gen["e_tables"]
        return edges, gfa, alt_len_from_gfa_text(gfa)
    if name == "A_utf8":
        ug = gen["utf8"][0]
        return ug.edges, ug.gfa_text, dict(ug.alt)
    g = gen["graph"]
    return g.edges, g.gfa_text, dict(g.alt)


@pytest.fixture(scope="module")
def gen():
    return generate()


# ---------------------------------------------------------------------------------------------------- CPU


def test_generator_covers_the_grid(gen):
    """Every chrom length of 1 to 17 bytes starts at every byte alignment; starts and ends of every digit count
    from 1 to 10; names that cross a 32-byte bitmap word and a 1 KiB step; every batch is populated."""
    b = gen["batches"]
    for name in (*PLAIN, *IRREGULAR_NODES, *IRREGULAR_LINES, *OTHER):
        batch = gen["utf8"][1] if name == "A_utf8" else b[name]
        assert len(batch.lines) >= 4, name
    a_names = ["A_plain", *IRREGULAR_NODES]
    grid, starts, ends, cross32, cross1k = set(), set(), set(), 0, 0
    for bn in a_names:
        for off, nm in name_spans(b[bn].lines):
            chrom, last = nm.rsplit(":", 1)
            grid.add((len(chrom.encode()), off & 3))
            end = off + len(nm.encode())
            cross32 += (off >> 5) != ((end - 1) >> 5)
            cross1k += (off >> 10) != ((end - 1) >> 10)
            if "-" in last and bn in ("A_plain", "A_digits10"):
                v0, v1 = last.split("-")
                starts.add(len(v0))
                ends.add(len(v1))
    assert {(n, a) for n in range(1, 18) for a in range(4)} <= grid
    assert set(range(1, 11)) <= starts and set(range(1, 11)) <= ends
    assert cross32 > 100 and cross1k > 5
    # the utf8 chroms: a byte with bit 7 set at the end of chroms of 13, 14 and 15 bytes, at every alignment
    ugrid = {(len(nm.rsplit(":", 1)[0].encode()), off & 3) for off, nm in name_spans(gen["utf8"][1].lines)}
    assert {(n, a) for n in (13, 14, 15) for a in range(4)} <= ugrid
    # the plain batches hold plain names only; the node-irregular ones hold an irregular name in every line
    assert all(len(n.rsplit(":", 1)[0].encode()) <= 15 for _o, n in name_spans(b["A_plain"].lines))
    assert all(len(n.rsplit(":", 1)[0].encode()) >= 16 for _o, n in name_spans(b["A_chrom16"].lines))
    # column runs of the B family right at the windows
    runs24, runs712 = set(), set()
    for line in b["B_plain"].lines + b["B_wide"].lines:
        cols = line.rstrip("\n").split("\t")
        runs24.add(sum(len(c) + 1 for c in cols[1:4]))
        runs712.add(sum(len(c) + 1 for c in cols[6:12]) - (0 if len(cols) > 12 else 1))
    assert {30, 31, 32, 33, 34} <= runs24 and {62, 63, 64, 65, 66} <= runs712
    assert not b["B_no_final_newline"].raw.endswith(b"\n") and not b["E"].raw.endswith(b"\n")
    assert b["E"].size > 2_000_000 and gen["n_irr_d"] > 3


def test_generator_is_deterministic():
    a, b = generate(with_e=False), generate(with_e=False)
    assert all(a["batches"][n].lines == b["batches"][n].lines for n in a["batches"])


@pytest.mark.parametrize("name", ASCII_BATCHES)
def test_c_oracle_equals_python_oracle(gen, name):
    """The checker of the GPU part (the C oracle) against the Python oracle on every batch: counters, record
    counts and informative_aln.json."""
    from oracle import c_oracle as CO
    CO.ensure_built()
    batch = gen["batches"][name]
    edges, _gfa, alt = tables_for(gen, name)
    ct = CO.Tables(edges, alt)
    counts, stats, sv2, off, ln = CO.filter_counts(ct, batch.raw, d_over=batch.d_over, want_hits=True)
    lines = O.text_mode_lines(batch.raw.decode())
    want = O.filter_alignments(lines, edges, alt, d_over=batch.d_over)
    assert CO.counts_dict(ct, counts) == O.hit_counts(want)
    assert stats["n_records"] == len(lines) and (stats["n_hits"] > 0) == (name != "A_alt_absent")
    assert O.dumps_informative(_dict_from_tuples(ct.sv_ids, batch.raw, sv2, off, ln)) == O.dumps_informative(want)


def _dict_from_tuples(sv_ids, raw, sv2, off, ln):
    d = {}
    order = np.lexsort((sv2, off))
    for s2, o, n in zip(sv2[order].tolist(), off[order].tolist(), ln[order].tolist()):
        d.setdefault(sv_ids[s2 >> 1], [[], []])[s2 & 1].append(O.kept_text(raw[o:o + n].decode()))
    return d


def test_node_tables_agree_on_every_generated_name(gen):
    """svjg_tables_alt_node_len probes the name table and, for a plain name, the exact-key table the scan
    kernel probes: the two must agree (-2 otherwise), and an alt node's length is the GFA's."""
    from svjg import alnfilter
    for name in ("A_plain", "A_utf8"):
        edges, gfa, alt = tables_for(gen, name)
        t = alnfilter.Tables.from_memory(json.dumps(edges, ensure_ascii=False), gfa)
        try:
            seen = {n for key in edges for n in key.split("@")[0::2]}
            assert len(seen) > 200
            for n in seen:
                got = t.alt_node_len(n)                                   # raises where the tables disagree
                if n in alt:
                    assert got == alt[n], n
        finally:
            t.close()


# ---------------------------------------------------------------------------------------------------- GPU


@pytest.fixture(scope="module")
def dev(gen):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from svjg import alnfilter, capi
    from oracle import c_oracle as CO
    CO.ensure_built()
    tables = {}

    def get(name, flags=0):
        key = ("E" if name == "E" else "A_utf8" if name == "A_utf8" else "private", flags)
        if key not in tables:
            edges, gfa, alt = tables_for(gen, name)
            t = alnfilter.Tables.from_memory(json.dumps(edges, ensure_ascii=False), gfa).to_device(0)
            t.set_flags(flags)
            tables[key] = (t, CO.Tables(edges, alt))
        return tables[key]
    yield alnfilter, capi, CO, torch, get
    for t, _ct in tables.values():
        t.close()


def _tuples(r):
    return sorted(zip(r.hit_sv2.tolist(), r.hit_off.tolist(), r.hit_len.tolist()))


def _check(CO, t, ct, raw, res, d_over, want=None):
    """Counters, record / multi-node / hit counts and the multiset of hit tuples of `res` against the C oracle."""
    if want is None:
        want = CO.filter_counts(ct, raw, d_over=d_over, want_hits=True)
    counts, stats, sv2, off, ln = want
    assert t.sv_ids == ct.sv_ids
    assert (res.counts == counts).all()
    assert {k: res.stats[k] for k in stats} == stats
    assert _tuples(res) == sorted(zip(sv2.tolist(), off.tolist(), ln.tolist()))
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n in ASCII_BATCHES if n != "E"])
def test_batch_matches_the_c_oracle_and_takes_its_route(dev, gen, name):
    alnfilter, capi, CO, torch, get = dev
    batch = gen["batches"][name]
    raw = batch.raw
    t, ct = get(name)
    res = alnfilter.filter_host(t, raw, d_over=batch.d_over)
    want = _check(CO, t, ct, raw, res, batch.d_over)
    st = res.stats
    assert (st["n_hits"] > 0) == (name != "A_alt_absent")            # that batch's lines have no link: no hit
    if name in PLAIN:
        # the scan kernel keeps every line: none goes to the exact kernel (whose giant_line() also applies the
        # fast rules, so n_generic alone would not show a line that left the fast route)
        assert st["n_exact"] == 0 and st["n_generic"] == 0 and st["n_multi"] > 0, st
    elif name in IRREGULAR_NODES:
        assert st["n_exact"] == len(batch.lines) and st["n_generic"] == st["n_multi"] == len(batch.lines), st
    elif name in IRREGULAR_LINES:
        assert st["n_exact"] == len(batch.lines), st
    elif name == "D_rounds":
        assert st["n_generic"] == gen["n_irr_d"], st
    # the general routine for every line: the same result
    tg, _ = get(name, capi.FLAG_FORCE_GENERAL)
    forced = alnfilter.filter_host(tg, raw, d_over=batch.d_over)
    _check(CO, tg, ct, raw, forced, batch.d_over, want)
    assert forced.stats["n_generic"] == forced.stats["n_multi"]


@pytest.mark.gpu
def test_non_ascii_chroms_match_the_oracle(dev, gen):
    """The C oracle declines non-ASCII bytes: the Python oracle is the checker (counters and the stored lines)."""
    alnfilter, capi, CO, torch, get = dev
    ug, batch, _ = gen["utf8"]
    t, _ct = get("A_utf8")
    raw = batch.raw
    res = alnfilter.filter_host(t, raw)
    want = O.filter_alignments(batch.lines, ug.edges, ug.alt)
    assert want and {t.sv_ids[i]: tuple(int(x) for x in res.counts[i]) for i in range(t.num_sv) if res.counts[i].any()} \
        == O.hit_counts(want)
    got = _dict_from_tuples(t.sv_ids, raw, res.hit_sv2, res.hit_off, res.hit_len)
    assert {k: [sorted(v[0]), sorted(v[1])] for k, v in got.items()} == \
        {k: [sorted(v[0]), sorted(v[1])] for k, v in want.items()}
    assert res.stats["n_exact"] == res.stats["n_generic"] == 0 and res.stats["n_multi"] == len(batch.lines)


def _tune(capi, knob, value):
    capi.check(capi.lib.svjg_filter_tune(knob, value))


@pytest.mark.gpu
def test_interleaved_batch_on_every_route_and_knob(dev, gen):
    """E: host route, device-rendered JSON byte for byte, resident route; then both scan geometries, forced
    tile sizes and lines per tile.  Every knob goes back to 0 whatever happens."""
    alnfilter, capi, CO, torch, get = dev
    batch = gen["batches"]["E"]
    raw = batch.raw
    t, ct = get("E")
    want = CO.filter_counts(ct, raw, want_hits=True)
    res = alnfilter.filter_host(t, raw)
    _check(CO, t, ct, raw, res, 100, want)
    assert res.stats["n_generic"] > 0 and res.stats["n_multi"] > 3000
    # informative_aln.json rendered on the device
    res2, text = alnfilter.filter_json_host(t, raw)
    assert text is not None and (res2.counts == want[0]).all()
    expect = O.dumps_informative(_dict_from_tuples(ct.sv_ids, raw, want[2], want[3], want[4]))
    assert bytes(text) == expect.encode()
    # resident route
    d = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
    f = alnfilter.DeviceFilter(t, hit_cap=want[1]["n_hits"] + 8)
    f.reset()
    f.run(d)
    _check(CO, t, ct, raw, f.result(), 100, want)
    # launch geometry: the Geo8 instantiation, forced tile sizes (4992 exceeds Geo8's window), lines per tile
    runs = [(blocks, tile, 0) for blocks in (6, 8) for tile in (0, 1024, 2048, 3360, 4992) if not (blocks == 8 and tile > 3360)]
    runs += [(0, 0, 8), (0, 0, 64)]
    try:
        for blocks, tile, lines in runs:
            _tune(capi, capi.TUNE_SCAN_BLOCKS, blocks)
            _tune(capi, capi.TUNE_TILE_BYTES, tile)
            _tune(capi, capi.TUNE_TILE_LINES, lines)
            got = alnfilter.filter_host(t, raw)
            _check(CO, t, ct, raw, got, 100, want)
            assert got.stats["n_generic"] == res.stats["n_generic"], (blocks, tile, lines)
    finally:
        _tune(capi, capi.TUNE_TILE_BYTES, 0)
        _tune(capi, capi.TUNE_TILE_LINES, 0)
        _tune(capi, capi.TUNE_SCAN_BLOCKS, 0)
