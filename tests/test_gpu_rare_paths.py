"""GPU parity tests for the branches of the scan and diff paths that only run above thresholds the other parity tests stay
below: streamed scans with events and Rev B, more than 16 groups, a full bare-assert queue in k_classify, the capacity
limits, stale device bytes behind unterminated last lines, lines and statements beyond 64 KiB, the 64-slab maximum, the
resident diff, pairs too far apart to trace and several trace batches.

Each test first asserts that it reached its branch (slab count from the cut rule of launch_scan, bare-assert count against
the grid bound of k_classify, edit distances against the limits of k_diff_small and k_myers_trace), so that a change of a
threshold cannot quietly turn it into one more small-corpus test.  Then every output is compared with the CPU oracle, or,
where the oracle cannot run, with exact values built into the input."""
import random

import numpy as np
import pytest

import corpus_util as cu
import orc
import tosemscan as ts

pytestmark = pytest.mark.gpu

FLAGS = ts.SCAN_ASSERT_EVENTS | ts.SCAN_HEADER_EVENTS
STATS = ("n_lines", "n_assert", "n_headers", "n_fixture", "digest")
SLAB = 32 << 20             # arena bytes per slab of a streamed tsm_scan (launch_scan)
MAX_SLABS = 64              # tsm_ctx::kMaxSlabs
BQ_CAP = 1024               # bare asserts one block of k_classify defers
CLS_BLOCKS_PER_SM = 8       # 256-thread blocks per SM: an upper bound on the k_classify grid
SMALL_MAX_D = 127           # largest distance k_diff_small finishes
SMALL_MAX_MIDDLE = 4096     # largest middle (lines of both sides between common head and tail) it finishes
TRACE_MAX_D = 23168         # largest distance k_myers_trace traces: (D+1)(D+2)/2 <= 2^28
TRACE_BATCH = 1 << 28       # trace ints per k_myers_trace launch


# ------------------------------------------------------------------------------------------------ helpers
def slab_cuts(c):
    """First file of every slab of a streamed tsm_scan over corpus c: the cut rule of launch_scan."""
    n = c.n_files
    if n == 0:
        return []
    off = np.asarray(c.off[:n + 1], np.int64)
    slab = SLAB
    while int(off[n]) // slab + 1 > MAX_SLABS:
        slab *= 2
    cuts, nxt = [0], slab
    while True:
        i = int(np.searchsorted(off[1:n], nxt, "left")) + 1     # first file i >= 1 with off[i] >= nxt
        if i >= n:
            return cuts
        cuts.append(i)
        nxt = int(off[i]) + slab


def oracle_scan(c, rev_b=False, events=True):
    return orc.scan(c.arena, c.off, c.len, c.ext, c.grp, c.n_groups, events=events, rev_b=rev_b)


def check_scan(got, want, flags, what=""):
    """Every output of a scan against the oracle: per-file records, both tables, totals, both event streams."""
    for f in STATS:
        bad = np.nonzero(got["stats"][f] != want["stats"][f])[0]
        assert bad.size == 0, (what, f, bad[:10], got["stats"][bad[:5]], want["stats"][bad[:5]])
    assert np.array_equal(got["group_counts"], want["group_counts"]), what
    assert np.array_equal(got["global_counts"], want["global_counts"]), what
    st = want["stats"]
    assert got["totals"].tolist() == [int(st[k].astype(np.int64).sum()) for k in STATS[:4]], what
    for key, bit in (("assert_events", ts.SCAN_ASSERT_EVENTS), ("header_events", ts.SCAN_HEADER_EVENTS)):
        if flags & bit:
            a, b = got[key], want[key]
            assert len(a) == len(b), (what, key, len(a), len(b))
            for f in a.dtype.names:
                bad = np.nonzero(a[f] != b[f])[0]
                assert bad.size == 0, (what, key, f, bad[:5], a[bad[:5]], b[bad[:5]])


def same_results(a, b, what=""):
    assert sorted(a) == sorted(b), what
    for k in a:
        assert np.array_equal(a[k], b[k]), (what, k)


def scan_resident(s, c, flags):
    s.upload(c)
    s.scan_resident(flags)
    r = s.download(flags)
    assert s.last_launch_count() == 3                        # one slab: k_plan, k_scan, k_classify
    return r


def check_line_records(s, c, ngram=3):
    gb, gh, ge, gf, gn = s.line_hashes(c, ngram=ngram)
    ob, oh, oe, of_ = orc.line_records(c.arena, c.off, c.len, c.ext)
    assert np.array_equal(gb, ob)
    for name, a, b in (("hash", gh, oh), ("end", ge, oe), ("flag", gf, of_), ("ngram", gn, orc.ngram_hashes(oh, ob, ngram))):
        bad = np.nonzero(a != b)[0]
        assert bad.size == 0, (name, bad[:8], a[bad[:4]], b[bad[:4]])
    return gb, gh, ge, gf, gn


def check_statements(s, c):
    got = s.statements(c)
    want = orc.statements(c.arena, c.off, c.len)
    for a, b in zip(got, want):
        bad = np.nonzero(a != b)[0]
        assert a.shape == b.shape and bad.size == 0, (bad[:8], a[bad[:4]], b[bad[:4]])
    return got


def oracle_diff(a, b):
    return orc.diff_pairs_detail((a.arena, a.off, a.len, a.ext), (b.arena, b.off, b.len, b.ext))


def check_diff(got, want, what=""):
    add, rem, det = got
    wadd, wrem, wdet = want
    bad = np.nonzero((add != wadd) | (rem != wrem))[0]
    assert bad.size == 0, (what, bad[:5], add[bad[:5]], wadd[bad[:5]], rem[bad[:5]], wrem[bad[:5]])
    for f in det.dtype.names:
        bad = np.nonzero(det[f] != wdet[f])[0]
        assert bad.size == 0, (what, f, bad[:5], det[bad[:5]], wdet[bad[:5]])


def copy_diff(r):
    return tuple(np.array(x, copy=True) for x in r)


def numbered(tag, n, assert_every=0):
    """n distinct lines; every assert_every-th one is an assertion line."""
    return [(b"assert %s%06d\n" if assert_every and i % assert_every == 0 else b"%s%06d = 1\n") % (tag, i) for i in range(n)]


def n_assert_lines(lines):
    return sum(orc.is_assert_line(l.rstrip(b"\n")) for l in lines)


def generated_files(seed, nbytes):
    """(bytes, ext) of C4-shaped generated files adding up to at least nbytes."""
    c = ts.gen_corpus(seed, max(16, nbytes // 9000), size_law=1, pinned=False)
    out, tot = [], 0
    for i in range(c.n_files):
        out.append((c.file_bytes(i), int(c.ext[i])))
        tot += int(c.len[i])
        if tot >= nbytes:
            return out
    raise AssertionError("generator made fewer bytes than asked for")


# ------------------------------------------------------------------------------------------------ 1. streamed scan, events, Rev B
def streamed_event_corpus(seed=0x5EA1):
    """~90 MiB: generated files, with fuzz and edge files on both sides of every slab cut and a 33 MiB file behind the
    first cut (its slab is larger than SLAB)."""
    rng = random.Random(seed)
    edge, edge_ext, _ = cu.edge_corpus()
    filler = generated_files(seed, 56 << 20)
    big = b"".join(f for f, _ in generated_files(seed + 1, SLAB + (1 << 20)))[:SLAB + (1 << 20)]
    big += b"\nclass TailOfTheBigFile:\n    def test_tail(self):\n        assert tail == 1\n        assert tail"
    files, exts = [], []
    st = {"off": 0, "nxt": SLAB}

    def add(b, e):
        if files and st["off"] >= st["nxt"]:
            st["nxt"] = st["off"] + SLAB                    # a cut: b starts the next slab
        files.append(b)
        exts.append(e)
        st["off"] += (len(b) + 127) // 128 * 128

    def fuzz_until(end):
        k = 0
        while st["off"] < end:
            fz, fe, _ = cu.fuzz_corpus(rng.randrange(1 << 30), 12, 9000)
            for b, e in zip(fz, fe):
                add(b, int(e))
            add(edge[k % len(edge)], int(edge_ext[k % len(edge)]))
            k += 1

    def cluster():                                           # fuzz from ~96 KiB in front of the cut to 64 KiB behind it
        target = st["nxt"]
        for b, e in zip(edge, edge_ext):
            add(b, int(e))
        fuzz_until(target + (64 << 10))

    big_done = False
    for b, e in filler:
        if st["off"] + len(b) >= st["nxt"] - (96 << 10):
            cluster()
            if not big_done:
                add(big, 1)                                  # the next file is a cut: slab = cluster tail + big file
                big_done = True
                fuzz_until(st["off"] + (64 << 10))
        add(b, e)
    return ts.pack(files, exts, [i % 7 for i in range(len(files))], 7, pinned=True)


def test_streamed_scan_with_events_and_rev_b():
    c = streamed_event_corpus()
    cuts = slab_cuts(c)
    n_slabs = len(cuts)
    assert n_slabs >= 3 and 80 << 20 <= int(c.off[-1]) <= 100 << 20
    bounds = [int(c.off[i]) for i in cuts] + [int(c.off[-1])]
    assert max(b - a for a, b in zip(bounds, bounds[1:])) > SLAB and int(c.len.max()) > SLAB
    want_a = oracle_scan(c)
    want_b = oracle_scan(c, rev_b=True)
    for want in (want_a, want_b):                          # assertion and header events on both sides of every cut
        for key in ("assert_events", "header_events"):
            f = want[key]["file"].astype(np.int64)
            for cut in cuts[1:]:
                assert ((f >= cut - 8) & (f < cut)).any() and ((f >= cut) & (f < cut + 8)).any(), (key, cut)
    s = ts.Scanner(0, int(c.off[-1]) + 4096, c.n_files, 16)
    try:
        got = s.scan(c, FLAGS)
        assert s.last_launch_count() == 3 * n_slabs
        check_scan(got, want_a, FLAGS, "rev A")
        fl = FLAGS | ts.SCAN_REV_B
        got_b = s.scan(c, fl)
        assert s.last_launch_count() == 3 * n_slabs
        check_scan(got_b, want_b, fl, "rev B")
        res_b = scan_resident(s, c, fl)                      # the same corpus resident: one slab, identical results
        check_scan(res_b, want_b, fl, "resident rev B")
        same_results(res_b, got_b, "resident vs streamed")
    finally:
        s.close()


# ------------------------------------------------------------------------------------------------ 2. more than 16 groups
@pytest.mark.parametrize("n_groups", [16, 17, 300, 65535])
def test_more_than_16_groups(n_groups):
    rng = np.random.default_rng(n_groups)
    files, exts, _ = cu.fuzz_corpus(1000 + n_groups, 400, 6000)
    edge, edge_ext, _ = cu.edge_corpus()
    files, exts = files + edge, np.concatenate([exts, edge_ext])
    grp = rng.integers(0, n_groups, len(files)).astype(np.uint16)
    grp[::97] = n_groups - 1
    small = ts.pack(files, exts, grp, n_groups)
    big = ts.gen_corpus(0x7053454D0002 + n_groups, 10000, 0, 4096)
    big.grp[:] = rng.integers(0, n_groups, big.n_files).astype(np.uint16)
    big.grp[-1] = n_groups - 1
    big.n_groups = n_groups
    n_slabs = len(slab_cuts(big))
    assert n_slabs >= 2
    s = ts.Scanner(0, int(big.off[-1]) + 4096, big.n_files, n_groups)
    try:
        for c, streamed in ((small, False), (big, True)):
            want = oracle_scan(c)
            assert want["group_counts"][n_groups - 1].sum() > 0
            got = s.scan(c, FLAGS)
            assert s.last_launch_count() == 3 * (n_slabs if streamed else 1)
            check_scan(got, want, FLAGS, ("host", streamed))
            assert np.array_equal(got["group_counts"].sum(axis=0), got["global_counts"])
            res = scan_resident(s, c, FLAGS)
            check_scan(res, want, FLAGS, ("resident", streamed))
            assert np.array_equal(res["group_counts"].sum(axis=0), res["global_counts"])
    finally:
        s.close()


# ------------------------------------------------------------------------------------------------ 3. full bare-assert queue
BARE = [b"assert not x", b"assert a in b", b"assert a is not None", b"assert x == True", b"assert a == b", b"assert a != b",
        b"assert a <= b", b"assert a >= b", b"assert a < b", b"assert a > b", b"assert not q in r", b"assert q is not r in s",
        b"assert True", b"assert x", b"assert y, 'no operator'", b"assert t.u.v"]
OTHER = [b"EXPECT_EQ(a, b);", b"EXPECT_TRUE(x);", b"EXPECT_NEAR(a, b, 1e-3);", b"ASSERT_NE(p, q);"]


def test_full_bare_assert_queue():
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rng = random.Random(7)
    block, n_bare_block = [], 0
    for i in range(4000):
        if rng.random() < 0.9:
            line = b" " * rng.choice([0, 4, 8]) + rng.choice(BARE)
            n_bare_block += 1                               # "assert <expr>": decided by the operator pass
        else:
            line = b"  " + rng.choice(OTHER)
        block.append(line + rng.choice([b"\n", b"\n", b"\r\n"]))
    body = b"".join(block)
    reps = 600
    files = [body * 4 for _ in range(reps // 4)]
    n_bare = n_bare_block * reps
    assert n_bare > BQ_CAP * CLS_BLOCKS_PER_SM * sms and n_bare > 2_000_000
    c = ts.pack(files, [1 if i % 3 else 2 for i in range(len(files))], [i % 5 for i in range(len(files))], 5, pinned=True)
    want_a = oracle_scan(c)
    want_b = oracle_scan(c, rev_b=True)
    for w in (want_a, want_b):
        assert int(w["stats"]["n_assert"].astype(np.int64).sum()) == len(block) * reps
    s = ts.Scanner(0, int(c.off[-1]) + 4096, c.n_files, 16, max_events=len(block) * reps + 4096)
    try:
        for fl, want in ((0, want_a), (FLAGS, want_a), (ts.SCAN_REV_B, want_b), (FLAGS | ts.SCAN_REV_B, want_b)):
            check_scan(scan_resident(s, c, fl), want, fl, fl)
    finally:
        s.close()


# ------------------------------------------------------------------------------------------------ 4. capacity limits
K = 1000


def assert_file(n_assert, n_hdr=0, pad=0):
    return b"".join([b"def test_c%d(self):\n" % i for i in range(n_hdr)] + [b"    assert x == %d\n" % i for i in range(n_assert)] +
                    [b"y = 1\n"] * pad)


def inert_file(nbytes):
    return (b"x = 1\n" * (nbytes // 6 + 1))[:nbytes]


def expect_capacity(fn):
    with pytest.raises(ts.TsmError) as e:
        fn()
    assert e.value.status == -3


def test_capacity_limits():
    ok = ts.pack([assert_file(250, 10, 30) for _ in range(4)], [1] * 4)
    over = ts.pack([assert_file(250, 10, 30) for _ in range(4)] + [assert_file(1)], [1] * 5)
    hdr_ok = ts.pack([assert_file(5, K // 2), assert_file(0, K // 2)], [1, 1])
    hdr_over = ts.pack([assert_file(5, K // 2), assert_file(0, K // 2 + 1)], [1, 1])
    streamed_ok = ts.pack([assert_file(K - 1), inert_file(SLAB + 4096), assert_file(1)], [1, 1, 1], pinned=True)
    streamed_over = ts.pack([assert_file(K), inert_file(SLAB + 4096), assert_file(1)], [1, 1, 1], pinned=True)
    want = {}
    for name, c, n_assert, n_hdr in (("ok", ok, K, 40), ("over", over, K + 1, 40), ("hdr_ok", hdr_ok, 5, K),
                                     ("hdr_over", hdr_over, 5, K + 1), ("streamed_ok", streamed_ok, K, 0),
                                     ("streamed_over", streamed_over, K + 1, 0)):
        want[name] = oracle_scan(c)
        st = want[name]["stats"]
        assert (int(st["n_assert"].sum()), int(st["n_headers"].sum())) == (n_assert, n_hdr), name
    assert len(slab_cuts(streamed_over)) == 2 and slab_cuts(streamed_over)[1] == 2
    s = ts.Scanner(0, 40 << 20, 64, 4, max_events=K)
    try:
        def recovers():                                      # after every -3 the ctx gives correct results again
            check_scan(s.scan(ok, FLAGS), want["ok"], FLAGS, "after -3")
        for fl in (0, FLAGS, ts.SCAN_HEADER_EVENTS):
            check_scan(s.scan(ok, fl), want["ok"], fl, ("exactly K", fl))
        for fl in (0, ts.SCAN_ASSERT_EVENTS, FLAGS, FLAGS | ts.SCAN_REV_B):
            expect_capacity(lambda: s.scan(over, fl))
            recovers()
        s.upload(over)
        s.scan_resident(FLAGS)
        expect_capacity(lambda: s.download(FLAGS))
        recovers()
        # header events alone: many headers, few asserts
        for fl in (ts.SCAN_HEADER_EVENTS, FLAGS):
            check_scan(s.scan(hdr_ok, fl), want["hdr_ok"], fl, ("exactly K headers", fl))
            expect_capacity(lambda: s.scan(hdr_over, fl))
            recovers()
        for fl in (0, ts.SCAN_ASSERT_EVENTS):                # without header events K + 1 headers fit
            check_scan(s.scan(hdr_over, fl), want["hdr_over"], fl, ("K+1 headers, no header events", fl))
        # the overflow only in the second slab of a streamed scan
        for fl in (0, FLAGS):
            check_scan(s.scan(streamed_ok, fl), want["streamed_ok"], fl, ("streamed K", fl))
            assert s.last_launch_count() == 6
            expect_capacity(lambda: s.scan(streamed_over, fl))
            recovers()
        # host side: the caller's event array is one short
        n_aev = len(want["ok"]["assert_events"])
        expect_capacity(lambda: s.scan(ok, FLAGS, event_cap=n_aev - 1))
        recovers()
    finally:
        s.close()


# ------------------------------------------------------------------------------------------------ 5. stale device bytes
JUNK = [b"assert(", b"EXPECT_", b"TEST_F(", b"_CHECK", b"def ", b"class ", b"{", b"\n"]
PARTIAL = [b"asser", b"EXPECT", b"TEST_", b"_CHEC", b"TESTEQUA", b"de"]
BODY = [b"    assert x == 1\n", b"EXPECT_EQ(a, b);\n", b"TEST_F(A, b) {\n", b"def test_x(self):\n", b"class T:\n",
        b"  BOOST_CHECK(x);\n", b"y = 2\n", b"\r\n", b"  TESTEQUAL(a, b);\n", b"void testIt() {\n"]


def junk_bytes(rng, n, newlines):
    toks = JUNK if newlines else JUNK[:-1]
    out = bytearray()
    while len(out) < n:
        out += rng.choice(toks)
    return bytes(out[:n])


def partial_file(rng, size, partial):
    if size <= len(partial):
        return partial[len(partial) - size:]
    out = bytearray()
    while len(out) < size - len(partial):
        out += rng.choice(BODY)
    return bytes(out[:size - len(partial)]) + partial


def test_stale_device_bytes_are_never_read():
    rng = random.Random(5)
    sizes = [128 * k + r for r in range(128) for k in (0, 1, 33)]
    sizes += [x + d for x in (4096, 4096 + 240, 8192, 8192 + 240) for d in (-1, 0, 1)]
    tfiles = [partial_file(rng, sz, PARTIAL[i % len(PARTIAL)]) for i, sz in enumerate(sizes)]
    texts = [(1, 2, 3, 4, 5, 6)[i % 6] for i in range(len(tfiles))]
    junk_1m = [junk_bytes(rng, 1 << 20, nl) for nl in (True, False)]

    def with_junk_gaps(c):                                   # gap bytes (SPEC section 1) hold junk too
        for i in range(c.n_files):
            a, b = int(c.off[i]) + int(c.len[i]), int(c.off[i + 1])
            c.arena[a:b] = np.frombuffer(junk_1m[i % 2][:b - a], np.uint8)
        return c
    target = with_junk_gaps(ts.pack(tfiles, texts, [i % 3 for i in range(len(tfiles))], 3, pinned=True))
    # streamed: a pattern-free file first, so that the first slab ends among the target files
    lead = inert_file(SLAB - 300_000)
    streamed = with_junk_gaps(ts.pack([lead] + tfiles, [1] + texts, [0] + [i % 3 for i in range(len(tfiles))], 3, pinned=True))
    cuts = slab_cuts(streamed)
    assert len(cuts) == 2 and 1 < cuts[1] < streamed.n_files - 1
    cap = ((int(streamed.off[-1]) >> 20) + 2) << 20
    junk = ts.pack([junk_1m[i % 2] for i in range(cap >> 20)], [(1, 2, 4)[i % 3] for i in range(cap >> 20)], pinned=True)
    assert int(junk.off[-1]) == cap                          # the junk fills the whole device arena
    jolds = ts.pack([junk.file_bytes(i) for i in range(6)], [1] * 6)
    want = {fl: oracle_scan(streamed, rev_b=bool(fl & ts.SCAN_REV_B)) for fl in (FLAGS, FLAGS | ts.SCAN_REV_B)}
    want_t = oracle_scan(target)
    olds = ts.pack(tfiles, texts)
    news = ts.pack([ts.gen_edit(77 + i, f, 3.0) if i % 4 else tfiles[(i * 7) % len(tfiles)] for i, f in enumerate(tfiles)], texts)
    want_d = oracle_diff(olds, news)
    outs = []
    for fresh in (False, True):
        s = ts.Scanner(0, cap, max(junk.n_files, streamed.n_files), 16)
        try:
            out = {}
            for fl in (FLAGS, FLAGS | ts.SCAN_REV_B):
                if not fresh:
                    s.scan(junk, FLAGS)
                out["streamed", fl] = s.scan(streamed, fl)
                assert s.last_launch_count() == 6
                check_scan(out["streamed", fl], want[fl], fl, ("streamed", fresh, fl))
                if not fresh:
                    s.scan(junk, 0)
                out["resident", fl] = scan_resident(s, streamed, fl)
                check_scan(out["resident", fl], want[fl], fl, ("resident", fresh, fl))
            if not fresh:
                s.scan(junk, 0)
            out["resident_target"] = scan_resident(s, target, FLAGS)
            check_scan(out["resident_target"], want_t, FLAGS, ("resident target", fresh))
            if not fresh:                                    # large junk calls first: the pool hands back their used slots
                s.line_hashes(junk)
            out["lines"] = check_line_records(s, target)
            if not fresh:
                s.statements(junk)
            out["stmts"] = check_statements(s, target)
            if not fresh:
                s.diff_pairs(jolds, jolds, detail=True)
            out["diff"] = s.diff_pairs(olds, news, detail=True)
            check_diff(out["diff"], want_d, ("diff", fresh))
            outs.append(out)
        finally:
            s.close()
    for k in outs[0]:                                        # and the same as a fresh context, output for output
        a, b = outs[0][k], outs[1][k]
        if isinstance(a, dict):
            same_results(a, b, k)
        else:
            assert all(np.array_equal(x, y) for x, y in zip(a, b)), k


# ------------------------------------------------------------------------------------------------ 6. long lines, large statements
def long_line_files():
    files, exts = [], []
    for nl in (b"\n", b"\r\n"):
        for n in (65534, 65535, 65536, 70000):               # T without '(': stmt_len saturates from 65 535 on
            files.append(b"def test_long(self):\n" + b"assert " + b"v" * (n - 7) + nl + b"    assert short == 1" + nl)
            pad = b"a or b " * (n // 7 + 1)
            files.append(b"  assert " + pad[:n - 16] + b" == True" + nl + b"assert x" + nl)
            files.append(b"    assert q != " + b"w" * (n - 16) + nl + b"assert tail < 2")
            exts += [1, 1, 1]
        for n in (65534, 65535, 65536, 70006):               # identifier run from `assert` to '(': ident_len saturates, <other>
            files.append(b"assert" + b"y" * (n - 6) + b"(q)" + nl + b"x = 1" + nl)
            exts.append(2)
        files.append(b"TEST_F(Suite, " + b"n" * 70000 + b") {" + nl + b"  EXPECT_EQ(" + b"a, " * ((1 << 20) // 3) + b"b);" + nl
                     + b"}" + nl)                            # a 1 MiB EXPECT_EQ( line and a 70 kB header line
        exts.append(3)
        files.append(b"public class LongTest {" + nl + b"  @Test public void testLong() {" + nl +
                     b"    assertEquals(a, " + b"b" * 70000 + b");" + nl + b"    assertTrue(" + b"c && " * 14000 + b"d);" + nl +
                     b"  }" + nl + b"}" + nl)                # Rev-B Java full statements longer than 64 KiB
        exts.append(4)
        files.append(b"BOOST_AUTO_TEST_CASE(Long) {" + nl + b"  BOOST_CHECK(" + b"x == " * 14000 + b"1);" + nl + b"}" + nl)
        exts.append(2)
    return files, exts


def test_long_lines_and_saturated_lengths():
    files, exts = long_line_files()
    c = ts.pack(files, exts, [i % 2 for i in range(len(files))], 2)
    s = ts.Scanner(0, 1 << 24, 1024, 16)
    try:
        for fl in (FLAGS, FLAGS | ts.SCAN_REV_B):
            want = oracle_scan(c, rev_b=bool(fl & ts.SCAN_REV_B))
            ev = want["assert_events"]
            assert (ev["stmt_len"] == 65535).sum() >= 16 and (ev["ident_len"] == 65535).sum() >= 6
            assert ((ev["ident_len"] == 65535) & (ev["cat"] == 127)).sum() >= 6
            assert (want["header_events"]["line_len"] > 70000).any()
            check_scan(s.scan(c, fl), want, fl, fl)
            check_scan(scan_resident(s, c, fl), want, fl, ("resident", fl))
        want_b = oracle_scan(c, rev_b=True)["assert_events"]
        assert ((want_b["stmt_len"] == 65535) & (np.asarray(exts)[want_b["file"]] == 4)).sum() >= 4
        check_line_records(s, c)
        check_statements(s, c)
        news = [f.replace(b"vvvv" + b"\n", b"vvvX\nassert new\n", 1).replace(b"b);", b"c);", 1) + b"added\n" for f in files]
        a, b = ts.pack(files, exts), ts.pack(news, exts)
        check_diff(s.diff_pairs(a, b, detail=True), oracle_diff(a, b))
    finally:
        s.close()


# ------------------------------------------------------------------------------------------------ 7. 64 slabs
def test_64_slab_maximum():
    """An arena of 2 030 MiB (4 KiB files) is cut into exactly 64 slabs: every slab event and slab record of the ctx is used.
    Costs about 2 GB of pinned host memory and 2 GB of HBM, plus the multi-threaded oracle over every file."""
    n = 2030 * 256
    c = ts.gen_corpus(0x7053454D0040, n, 0, 4096, n_groups=9)
    assert 2017 << 20 <= int(c.off[-1]) <= 2047 << 20
    n_slabs = len(slab_cuts(c))
    assert n_slabs == MAX_SLABS
    s = ts.Scanner(0, int(c.off[-1]), n, 16)
    try:
        got = s.scan(c, 0)
        assert s.last_launch_count() == 3 * n_slabs == 192
    finally:
        s.close()
    mt = orc.MtScanner(0, 16)
    try:
        want = mt.scan(c.arena, c.off, c.len, c.ext, c.grp, 9)
        check_scan(got, want, 0)
    finally:
        mt.close()


# ------------------------------------------------------------------------------------------------ 8. resident diff
def c5_pairs(seed, n, cap):
    base = ts.gen_corpus(0x7053454D0005 + seed, n, size_law=1, pinned=False)
    olds = [base.file_bytes(i)[:cap] for i in range(n)]
    return olds, [ts.gen_edit(1000 + seed * 7919 + i, o, 6.0) for i, o in enumerate(olds)]


def leftover_pairs():
    """Pairs k_diff_small leaves over: distance above 127, or a middle of more than 4 096 lines."""
    olds, news = [], []
    for total, d in ((1300, 128), (2000, 300), (1800, 700)):  # d deletions spread over the file
        o = numbered(b"p", total, 5)
        step = total // d
        olds.append(b"".join(o))
        news.append(b"".join(l for i, l in enumerate(o) if not (i % step == 1 and i // step < d)))
    for total in (4100, 6000):                               # 2 edits at the ends of a long middle
        half = total // 2
        olds.append(b"head\n" * 40 + b"first old\n" + b"".join(numbered(b"m", half - 2)) + b"last old\n" + b"tail\n" * 40)
        news.append(b"head\n" * 40 + b"first new\n" + b"".join(numbered(b"m", total - half - 2)) + b"assert last_new\n" + b"tail\n" * 40)
    olds.append(b"".join(numbered(b"o", 400, 3)))            # unrelated sides
    news.append(b"".join(numbered(b"n", 350, 4)))
    return olds, news


def test_resident_diff():
    co, cn = c5_pairs(11, 300, 65536)
    lo, ln = leftover_pairs()
    olds, news = co + lo, cn + ln
    exts = [(1, 2, 4)[i % 3] for i in range(len(olds))]
    a, b = ts.pack(olds, exts, pinned=True), ts.pack(news, exts, pinned=True)
    want = oracle_diff(a, b)
    D = want[0] + want[1]
    nl = len(lo)
    assert (D[-nl:-3] > SMALL_MAX_D).all() and (D[-1] > SMALL_MAX_D)
    assert all(o.count(b"\n") + n.count(b"\n") - 4 * 40 > SMALL_MAX_MIDDLE for o, n in zip(lo[-3:-1], ln[-3:-1]))
    s = ts.Scanner(0, 1 << 22, 1024, 4)
    try:
        s.diff_upload(a, b)
        runs = []
        for _ in range(3):                                   # the result buffers are pinned and reused: copy them
            runs.append(copy_diff(s.diff_resident(True)))
            assert s.diff_last_ms()[2] > 0                   # k_myers / k_myers_trace ran for the left-over pairs
        for r in runs:
            check_diff(r, want, "resident")
            check_diff(r, copy_diff(runs[0]), "repeat")
        check_diff(s.diff_pairs(a, b, detail=True), want, "host path")
        add, rem = s.diff_resident(False)
        assert np.array_equal(add, want[0]) and np.array_equal(rem, want[1])
        # a second upload with another pair count replaces the first
        k = 57
        a2, b2 = ts.pack(olds[-k:], exts[-k:], pinned=True), ts.pack(news[-k:], exts[-k:], pinned=True)
        s.diff_upload(a2, b2)
        r2 = copy_diff(s.diff_resident(True))
        assert len(r2[0]) == k
        check_diff(r2, tuple(w[-k:] for w in want), "second upload")
    finally:
        s.close()
    fresh = ts.Scanner(0, 1 << 20, 16, 1)
    try:
        out = np.zeros(4, np.int64)
        assert ts.lib().tsm_diff_resident(fresh._ctx, ts._p(out), ts._p(out), None, None) == -6
    finally:
        fresh.close()


# ------------------------------------------------------------------------------------------------ 9. distant pairs, trace batches
def test_untraced_distant_pairs():
    """LCS = 0 (disjoint distinct lines): added = |new|, removed = |old|, one mod hunk.  D = 23 168 is traced (assertion lines
    of each side counted), D = 23 169 is not (-1 / -1).  Ordinary pairs in the same call are checked against the oracle."""
    far = []
    for n_old, n_new in ((11584, 11584), (11585, 11584)):
        o, n = numbered(b"old", n_old, 7), numbered(b"new", n_new, 5)
        far.append((b"".join(o), b"".join(n), n_old, n_new, n_assert_lines(o), n_assert_lines(n)))
    assert [x[2] + x[3] for x in far] == [TRACE_MAX_D, TRACE_MAX_D + 1]
    assert far[0][4] > 0 and far[0][5] > 0
    co, cn = c5_pairs(12, 40, 20000)
    small_o, small_n = b"".join(numbered(b"a", 150, 3)), b"".join(numbered(b"b", 130, 4))   # disjoint, traced: the same rule
    olds = co[:20] + [far[0][0], small_o] + co[20:] + [far[1][0]]
    news = cn[:20] + [far[0][1], small_n] + cn[20:] + [far[1][1]]
    exts = [1] * len(olds)
    far_at = [20, len(olds) - 1]
    s = ts.Scanner(0, 1 << 22, 1024, 4)
    try:
        add, rem, det = s.diff_pairs(ts.pack(olds, exts), ts.pack(news, exts), detail=True)
    finally:
        s.close()
    for i, (_, _, n_old, n_new, a_old, a_new) in zip(far_at, far):
        traced = n_old + n_new <= TRACE_MAX_D
        assert (int(add[i]), int(rem[i])) == (n_new, n_old)
        assert tuple(int(x) for x in det[i]) == (0, 0, 1) + ((a_new, a_old) if traced else (-1, -1)), (i, det[i])
    keep = [i for i in range(len(olds)) if i not in far_at]
    ko, kn = ts.pack([olds[i] for i in keep], exts[:len(keep)]), ts.pack([news[i] for i in keep], exts[:len(keep)])
    want = oracle_diff(ko, kn)
    check_diff((add[keep], rem[keep], det[keep]), want, "ordinary pairs")
    j = keep.index(21)                                       # the small disjoint pair: one mod hunk in the oracle too
    assert tuple(int(x) for x in want[2][j])[:3] == (0, 0, 1) and int(want[0][j] + want[1][j]) == 280
    assert (int(want[2][j]["added_assert"]), int(want[2][j]["removed_assert"])) == (
        n_assert_lines(numbered(b"b", 130, 4)), n_assert_lines(numbered(b"a", 150, 3)))


def test_trace_in_several_batches():
    """Left-over pairs with D of 6 000 - 8 000 whose trace tables add up to more than 2^28 ints: k_myers_trace runs in
    several batches.  Every pair's detail against the oracle."""
    rng = random.Random(3)
    olds, news = [], []
    for p in range(14):
        o = numbered(b"q%02d_" % p, 10000, 6)
        n = []
        for i, l in enumerate(o):
            r = rng.random()
            if r < 0.5:
                continue                                     # deleted
            if r < 0.6:
                n.append(b"assert ins%02d_%06d\n" % (p, i))
            elif r < 0.7:
                n.append(b"ins%02d_%06d = 2\n" % (p, i))
            n.append(l)
        olds.append(b"".join(o))
        news.append(b"".join(n))
    exts = [1] * len(olds)
    a, b = ts.pack(olds, exts), ts.pack(news, exts)
    want = oracle_diff(a, b)
    D = (want[0] + want[1]).astype(np.int64)
    assert D.min() > SMALL_MAX_D and 5000 <= D.min() and D.max() <= 8000
    need = (D + 1) * (D + 2) // 2
    assert int(need.sum()) > TRACE_BATCH
    batches, tot = 1, 0                                      # the batch rule of diff_core
    for x in need.tolist():
        if tot and tot + x > TRACE_BATCH:
            batches, tot = batches + 1, 0
        tot += x
    assert batches >= 2
    s = ts.Scanner(0, 1 << 22, 1024, 4)
    try:
        check_diff(s.diff_pairs(a, b, detail=True), want, "batched trace")
    finally:
        s.close()
