"""CPU tests: the oracle against the reference's golden vectors and against independent
pure-Python restatements of docs/SPEC.md (no GPU needed)."""
import json
import os
import random

import numpy as np
import pytest

import corpus_util as cu
import orc

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
M61 = (1 << 61) - 1
MASK = (1 << 64) - 1


def py_bytes_hash(b: bytes) -> int:
    """SPEC section 3 with Python big integers."""
    h = int.from_bytes(b, "little") % M61
    x = h ^ ((len(b) * 0x9E3779B97F4A7C15) & MASK)
    x ^= x >> 30
    x = (x * 0xBF58476D1CE4E5B9) & MASK
    x ^= x >> 27
    x = (x * 0x94D049BB133111EB) & MASK
    x ^= x >> 31
    return x


def py_lines(data: bytes):
    """SPEC section 2."""
    if not data:
        return []
    parts = data.split(b"\n")
    if parts[-1] == b"":
        parts.pop()
    return parts


def test_hash_matches_bigint_definition():
    rng = random.Random(1)
    cases = [b"", b"\x00", b"\x00\x00", b"a", b"\xff" * 61, b"\xff" * 122, bytes(range(256)),
             b"x" * 8, b"x" * 7, b"x" * 9, b"\xff" * 7 + b"\x1f"]
    cases += [bytes(rng.randrange(256) for _ in range(rng.randrange(0, 300))) for _ in range(300)]
    for c in cases:
        assert orc.bytes_hash(c) == py_bytes_hash(c), c
    assert orc.line_hash(b"abc\r") == py_bytes_hash(b"abc")
    assert orc.line_hash(b"abc\r\r") == py_bytes_hash(b"abc\r")
    assert orc.line_hash(b"\r") == py_bytes_hash(b"")
    # the modulus value itself must canonicalise to 0
    assert orc.bytes_hash(b"\xff" * 7 + b"\x1f") == py_bytes_hash(b"\xff" * 7 + b"\x1f")


def test_line_splitting_and_counts():
    for data, want in [(b"", 0), (b"a\n", 1), (b"a\nb", 2), (b"\n\n", 2), (b"\n", 1), (b"a", 1), (b"\r\n", 1)]:
        arena, off, ln = orc.pack([data])
        res = orc.scan(arena, off, ln, np.array([1], np.uint8), np.array([0], np.uint16), 1, line_hashes=True)
        assert res["stats"]["n_lines"][0] == want == len(py_lines(data))
        assert [int(h) for h in res["line_hash"]] == [py_bytes_hash(l[:-1] if l.endswith(b"\r") else l) for l in py_lines(data)]
        assert int(res["stats"]["digest"][0]) == sum(int(h) for h in res["line_hash"]) & MASK


def test_g4_statement_category_golden():
    """Golden G4: every (statement, category) pair of the five Rev-A sheets of ML-Testing-v1.xlsx."""
    rows = json.load(open(os.path.join(GOLD, "g4_statement_category.json")))
    ledger = json.load(open(os.path.join(GOLD, "ledger.json")))["G4"]
    known_misses = {(m["statement"], m["sheet_says"]) for m in ledger["misses"]}
    hit = tot = 0
    for r in rows:
        st = r["statement"].encode("utf-8")
        # S4: statements are already truncated and stripped
        assert orc.statement(st) == st
        got = orc.category_string(st)
        tot += r["rows"]
        if got == r["category"]:
            hit += r["rows"]
        else:
            assert (r["statement"], r["category"]) in known_misses, (r, got)
    assert [hit, tot] == ledger["category_rule_rows"] == [11954, 11981]


def test_classify_rules():
    name = orc.category_string
    assert name(b"EXPECT_EQ") == "assertEqual" and name(b"ASSERT_NEAR") == "assertAlmostEqual"
    assert name(b"EXPECT_STREQ") == "" and name(b"EXPECT_") == "" and name(b"else ASSERT_EQ") == "assertEqual"
    assert name(b"EXPECT_THROW") == "assertRaises" and name(b"EXPECT_DOUBLE_EQ") == "assertDoubleEqual"
    assert name(b"assert") == "assertTrue" and name(b"assert agent") == "assertTrue"
    assert name(b"assert not agent.no_pull") == "assertNotEqual"
    assert name(b'assert "Schedule not found" in str') == "assertFalse"
    assert name(b'assert result == 0, "Repo did not pass Black formatting!"') == "assertEqual"
    assert name(b"assert x is not None") == "assertFalse"
    assert name(b"assert res.mapped == True") == "assertTrue"
    assert name(b"assert a <= b") == "assertLessEqual" and name(b"assert a >= b") == "assertGreaterEqual"
    assert name(b"assert a < b") == "assertLess" and name(b"assert a > b") == "assertGreater"
    assert name(b"assert a != b") == "assertNotEqual"
    assert name(b"self.assertEquals") == "assertEquals" and name(b"self.assert_") == "assertTrue"
    assert name(b"self.assertWeirdCustomThing") == "assertWeirdCustomThing"
    assert orc.classify(b"self.assertWeirdCustomThing")[0] == 127
    assert name(b"x.assert_called_once_with") == "assert_called_once_with"
    assert name(b"if") == "" and name(b"GPUAssert") == "" and name(b"") == "" and name(b'"""') == ""
    assert name(b"assert\tx") == "" and name(b"assertx") == "assertx"
    # every table name maps to its own id
    for i in range(1, 127):
        nm = orc.category_name(i)
        if nm:
            assert orc.classify(b"self." + nm.encode())[0] == i


def test_statement_truncation():
    assert orc.statement(b"   self.assertEqual(a, b)  ") == b"self.assertEqual"
    assert orc.statement(b"\tassert sys.version_info >= (3, 6)\r") == b"assert sys.version_info >="
    assert orc.statement(b"assert x") == b"assert x"
    assert orc.statement(b"(assert)") == b""
    assert orc.statement(b"   ") == b""


def test_header_rules_and_method_strings():
    hk, ms = orc.header_kind, orc.method_string
    # PY (SPEC section 5)
    assert hk(1, b"    def test_docker_agent_init(monkeypatch, runner_token):") == 1
    assert ms(1, b"    def test_docker_agent_init(monkeypatch, runner_token):") == b"test_docker_agent_init(monkeypatch,runner_token)"
    assert ms(1, b"def test_training_pipeline(config: Config, model_type: str, car_dir: str) \\") == \
        b"test_training_pipeline(config:Config,model_type:str,car_dir:str)\\"
    assert hk(1, b"parser.add_argument('-t', '--tested-skills', default=[])") == 1
    assert ms(1, b"parser.add_argument('-t', '--tested-skills', default=[])") == b"parser.add_argument('-t','--tested-skills',ault=[])"
    assert hk(1, b"class SkillTest(object):") == 1 and ms(1, b"class SkillTest(object):") == b"SkillTest(object)"
    assert hk(1, b"classifier = 3") == 0 and hk(1, b"x = class Foo") == 0 and hk(1, b"class\tT:") == 1
    assert ms(1, b"    async def test_x(self):") == b"asynctest_x(self)"
    # C family
    assert hk(2, b'      : sensor1_dst_("test"), sensor2_dst_("test"), fused_dst_("test") {') == 1
    assert ms(2, b'      : sensor1_dst_("test"), sensor2_dst_("test"), fused_dst_("test") {') == b': sensor1_dst_("test"'
    assert hk(2, b'    dst_manager->AddApp("test", fod_subsets, fod_subset_names);') == 0
    assert hk(2, b"  ~DSTEvidenceTest() {}") == 1 and ms(2, b"  ~DSTEvidenceTest() {}") == b"~DSTEvidenceTest("
    assert hk(2, b"TEST_F(DsmTest, Invalid) {") == 3 and ms(2, b"TEST_F(DsmTest, Invalid) {") == b"TEST_F(DsmTest, Invalid"
    assert hk(2, b"  TEST_F(DsmTest, Invalid) {") == 3
    assert ms(3, b"class NavigationLaneTest : public testing::Test {") == b"class NavigationLaneTest : public testing::Test"
    assert hk(2, b"  void CreateTestMapNode(unsigned int m, unsigned int n,") == 1
    assert hk(2, b'  EXPECT_EQ(latest_observed_msg_ptr->class_name(), "BlockerTest");') == 1
    assert hk(2, b"for (int i = 0; i < n; ++i) {") == 0
    assert hk(0, b"TEST_F(A, B) {") == 0
    # Java
    assert ms(4, b"    public void testFactory() throws Exception {") == b"testFactory()throwsException{"
    assert ms(4, b"public class MapDecodeTest {") == b"MapDecodeTest{"
    assert ms(4, b"  @Test public void testDoubleInitialize() throws Exception {") == b"@TesttestDoubleInitialize()throwsException{"


def test_g3_correlate_table_from_the_taxonomy_fixture():
    """RQs/RQ3/tests_correlate_rq3.csv (20 strategies x 21 properties): the flag columns rebuilt from the committed
    taxonomy columns (tests/golden/taxonomy_min.csv.gz), reduced by the oracle, formatted like the shipped cells
    ("repo:(p%), " with p a Python float of 2 decimals, "0" for a pairing no case has): 394 of 420 cells bit-identical."""
    import csv
    import gzip
    import io
    d = np.load(os.path.join(GOLD, "g3_reduce.npz"))
    rows = list(csv.DictReader(io.StringIO(gzip.open(os.path.join(GOLD, "taxonomy_min.csv.gz"), "rb").read().decode("utf-8"), newline="")))
    repos = [str(x) for x in d["repo_names"]]
    rid = {r: i for i, r in enumerate(repos)}
    cases = sorted({r["Cases"] for r in rows}, key=lambda s: (len(s), s))
    cid = {c: i for i, c in enumerate(cases)}
    rcol, rval = [str(x) for x in d["correlate_row_column"]], [str(x) for x in d["correlate_row_value"]]
    labels = [set(str(x).split("|")) for x in d["correlate_col_labels"]]
    nr, nc = len(rcol), len(labels)
    flags = np.zeros((len(rows), nr * nc), np.uint8)
    for i, r in enumerate(rows):
        pr = [(r["Data"].strip() in lab) or (r["Model"].strip() in lab) for lab in labels]
        for j in range(nr):
            if r[rcol[j]].strip() == rval[j]:
                flags[i, j * nc:(j + 1) * nc] = pr
    repo = np.array([rid[r["Repo"]] for r in rows], np.int32)
    case = np.array([cid[r["Cases"]] for r in rows], np.int32)
    out, cpr = orc.reduce(flags, repo, case, len(repos), len(cases))
    assert np.array_equal(out, d["oracle_correlate_distinct"])
    order = [str(x) for x in d["correlate_repo_order"]]
    ok, want = d["correlate_cell_reproduces"], d["want_correlate_cells"]
    assert ok.shape == (20, 21) and int(ok.sum()) == 394 and int((ok.sum(axis=1) == 21).sum()) == 5
    for j in range(nr):
        for q in range(nc):
            dd = [int(out[j * nc + q, rid[n]]) for n in order]
            cell = "0" if not any(dd) else "".join("%s:(%s%%), " % (n, repr(round(100.0 * v / int(cpr[rid[n]]), 2))) for n, v in zip(order, dd))
            assert (cell == str(want[j][q])) == bool(ok[j, q]), (j, q)
            # the two other shipped layouts of the same counts (tests_correlate_rq4.csv, tests_combined_correlate_rq3.csv)
            tex = "".join("$%s:%s\\%%$, " % (n, repr(round(100.0 * v / int(cpr[rid[n]]), 2))) for n, v in zip(order, dd) if v) or "0"
            assert (tex == str(d["want_correlate_tex_cells"][j][q])) == bool(d["correlate_tex_cell_reproduces"][j, q]), (j, q)
            assert (str(sum(dd)) == str(d["want_correlate_count_cells"][j][q])) == bool(d["correlate_count_cell_reproduces"][j, q]), (j, q)
    assert int(d["correlate_tex_cell_reproduces"].sum()) == 394 and int(d["correlate_count_cell_reproduces"].sum()) == 382


def test_g3_merged_row_tables():
    """tests_correlate_{FileError,RuntimeError,assertion,logical}.csv: the correlate layout for the merged strategy rows,
    rebuilt from the committed flag matrix (strategy flag AND property flag), 78 of 84 cells bit-identical."""
    d = np.load(os.path.join(GOLD, "g3_reduce.npz"))
    names = [str(x) for x in d["flag_names"]]
    repos = [str(x) for x in d["repo_names"]]
    order = [str(x) for x in d["correlate_repo_order"]]
    props = ["p:" + {"Distribution": "Data Distribution", "Validity": "Data Validity", "Relation": "Data Relation",
                     "Feature Importance": "Features Importance", "Restoration": "Data Restoration and Recoverability",
                     "Concurrency": "Concurrency and Parallelism", "uncertainty": "Uncertainty", "Data Loss": "Data Migration Loss and Corruption",
                     "Bias": "Bias and Fairness", "Security": "Security and Privacy", "Uniqueness": "Data Uniqueness",
                     "Timeliness": "Data Timeliness", "integration": "Data Integration Integrity",
                     "Compatibility": "Compatibility and Portability"}.get(str(c), str(c)) for c in d["correlate_col_names"]]
    F = d["flags"]
    cols = []
    for srow in d["merged_strategy_rows"]:
        for pname in props:
            cols.append(F[:, names.index(str(srow))] & F[:, names.index(pname)])
    out, cpr = orc.reduce(np.stack(cols, axis=1).astype(np.uint8), d["repo"], d["case_id"], len(repos), int(d["case_id"].max()) + 1)
    assert np.array_equal(out, d["oracle_merged_distinct"])
    ok, want = d["merged_cell_reproduces"], d["want_merged_cells"]
    for j in range(ok.shape[0]):
        for q in range(ok.shape[1]):
            dd = [int(out[j * ok.shape[1] + q, repos.index(n)]) for n in order]
            cell = "0" if not any(dd) else "".join("%s:(%s%%), " % (n, repr(round(100.0 * v / int(cpr[repos.index(n)]), 2))) for n, v in zip(order, dd))
            assert (cell == str(want[j][q])) == bool(ok[j, q]), (j, q)
    assert [int(x) for x in ok.sum(axis=1)] == [21, 16, 21, 20]


def test_g3_reduce_golden():
    """Golden G3: RQs/taxonomy_test2.csv -> tests_strategy_rq32.csv / tests_methods_v2.csv."""
    d = np.load(os.path.join(GOLD, "g3_reduce.npz"))
    out, cpr = orc.reduce(d["flags"], d["repo"], d["case_id"], len(d["repo_names"]), int(d["case_id"].max()) + 1)
    assert np.array_equal(out, d["oracle_distinct"]) and np.array_equal(cpr, d["oracle_cases_per_repo"])
    assert cpr.tolist() == [181, 164, 142, 160, 124, 100, 90, 216, 273] and cpr.sum() == 1450
    ok = d["strategy_cell_reproduces"]
    assert int(ok.sum()) == 171 and ok.size == 171          # every shipped cell (with the recovered Error_Type merges)
    # re-derive the shipped cells (rounded twice: SPEC section 9) wherever the ledger says they reproduce
    for j in range(ok.shape[0]):
        for k in range(ok.shape[1]):
            if ok[j, k]:
                v = round(round(100.0 * out[j, k] / cpr[k], 4) / 1.1, 4)
                s = ("%.4f" % v).rstrip("0").rstrip(".") or "0"
                assert s == str(d["want_strategy_cells"][j][k])
    ns = ok.shape[0]
    rep = d["method_reproduces"].astype(bool)
    tot = out[ns:ns + len(rep)].sum(axis=1)
    assert np.array_equal(tot[rep], d["want_method_total_cases"][rep]) and int(rep.sum()) == 11
    # RQ3 property table (tests_prop_rq3.csv): 100 * distinct / 216 (Apollo's case count), 17 of 21 columns exact
    pok = d["property_cell_reproduces"]
    assert pok.shape == (21, 9) and int(pok.sum()) == 172 and int((pok.sum(axis=1) == 9).sum()) == 17
    p0 = ns + len(rep)
    denom = int(cpr[list(d["repo_names"]).index("Apollo")])
    assert denom == 216
    for j in range(pok.shape[0]):
        for k in range(pok.shape[1]):
            if pok[j, k]:
                s = ("%.4f" % round(100.0 * out[p0 + j, k] / denom, 4)).rstrip("0").rstrip(".") or "0"
                assert s == str(d["want_property_cells"][j][k])


def test_lcs_oracle_against_bruteforce():
    rng = random.Random(7)

    def brute(a, b):
        dp = [[0] * (len(b) + 1) for _ in range(len(a) + 1)]
        for i in range(len(a)):
            for j in range(len(b)):
                dp[i + 1][j + 1] = dp[i][j] + 1 if a[i] == b[j] else max(dp[i][j + 1], dp[i + 1][j])
        return dp[-1][-1]
    for _ in range(200):
        a = [rng.randrange(6) for _ in range(rng.randrange(0, 30))]
        b = [rng.randrange(6) for _ in range(rng.randrange(0, 30))]
        assert orc.lcs(np.array(a, np.uint64), np.array(b, np.uint64)) == brute(a, b)


def test_diff_script_distance_and_hunks():
    """SPEC section 8: D equals n + m - 2 LCS, and the hunk bookkeeping on hand-checked cases."""
    rng = random.Random(11)
    for _ in range(300):
        a = [rng.randrange(5) for _ in range(rng.randrange(0, 25))]
        b = [rng.randrange(5) for _ in range(rng.randrange(0, 25))]
        D, det = orc.diff_script(a, b)
        assert D == len(a) + len(b) - 2 * orc.lcs(np.array(a, np.uint64), np.array(b, np.uint64))
        # every hunk has at least one edit; a mod hunk has at least two
        assert det["hunks_add"] + det["hunks_del"] + 2 * det["hunks_mod"] <= D or D == 0
        assert (D == 0) == (det["hunks_add"] + det["hunks_del"] + det["hunks_mod"] == 0)
    cases = [([1, 2, 3], [1, 2, 3], (0, 0, 0)), ([1, 2, 3], [1, 3], (0, 1, 0)), ([1, 3], [1, 2, 3], (1, 0, 0)),
             ([1, 2, 3], [1, 9, 3], (0, 0, 1)), ([], [5, 6], (1, 0, 0)), ([5, 6], [], (0, 1, 0)),
             ([1, 2, 3, 4, 5], [1, 8, 3, 9, 5], (0, 0, 2)), ([1, 2, 3, 4, 5, 6, 7], [2, 3, 4, 5, 6, 7, 8], (1, 1, 0))]
    for a, b, want in cases:
        D, det = orc.diff_script(a, b)
        assert (det["hunks_add"], det["hunks_del"], det["hunks_mod"]) == want, (a, b, det)
    D, det = orc.diff_script([1, 2, 3, 4], [1, 7, 4], fa=[0, 1, 1, 0], fb=[0, 1, 0])
    assert D == 3 and det["removed_assert"] == 2 and det["added_assert"] == 1 and det["hunks_mod"] == 1


def test_statements_match_python_restatement():
    """SPEC section 10 against the three-line Python rule the golden G2 recall was measured with."""
    def py_statements(data):
        out, cur, depth = [], [], 0
        for line in data.split(b"\n"):
            s = line.strip(b" \t\r\x0b\x0c")
            if not s:
                continue
            cur.append(s)
            depth += s.count(b"(") - s.count(b")")
            if depth <= 0:
                out.append(b" ".join(cur))
                cur, depth = [], 0
        if cur:
            out.append(b" ".join(cur))
        return out
    files, _, _ = cu.edge_corpus()
    rng = random.Random(4)
    files = list(files) + [cu.fuzz_file(rng, rng.randrange(1, 3000), nl_rate=0.15) for _ in range(60)]
    files += [b"EXPECT_EQ(\n    box1.DebugString(),\n    \"aabox2d ( x )\");\nfoo();\n", b"a(\n\n b(\n))\n)\n)\nx\n", b"((((\n"]
    for f in files:
        assert orc.statement_texts(f) == py_statements(f), f[:60]
    assert orc.statement_texts(files[-3]) == [b'EXPECT_EQ( box1.DebugString(), "aabox2d ( x )");', b"foo();"]


def test_g2_recall_ledger():
    """Golden G2 (ML-Analysis-v4.xlsx body statements): recall recorded by tools/make_golden.py with the oracle."""
    g2 = json.load(open(os.path.join(GOLD, "ledger.json")))["G2"]["subjects"]
    assert g2["Apollo"]["rows_recalled"] == [5644, 5947] and g2["DeepSpeech2"]["rows_recalled"] == [1657, 1813]
    assert g2["autokeras"]["rows_recalled"] == [351, 406] and g2["Nupic"]["rows_recalled"][0] >= 3934


def test_scan_on_edge_corpus_matches_python_restatement():
    files, exts, grps = cu.edge_corpus()
    arena, off, ln = orc.pack(files)
    res = orc.scan(arena, off, ln, exts, grps, 3)
    for i, f in enumerate(files):
        lines = py_lines(f)
        st = res["stats"][i]
        assert st["n_lines"] == len(lines)
        if exts[i]:
            want = sum(1 for l in lines if b"assert" in l.lower() or b"EXPECT_" in l)
            assert st["n_assert"] == want, (i, f[:40])
        else:
            assert st["n_assert"] == 0 and st["n_headers"] == 0
    ev = res["assert_events"]
    assert len(ev) == int(res["stats"]["n_assert"].sum()) == int(res["global_counts"].sum())
    assert np.array_equal(res["group_counts"].sum(axis=0), res["global_counts"])
    # events are in canonical order and their statement hash is the hash of the statement bytes
    key = ev["file"].astype(np.int64) << 32 | ev["line_off"]
    assert np.all(np.diff(key) > 0)
    for e in ev[:200]:
        f = files[e["file"]]
        t = f[e["stmt_off"]:e["stmt_off"] + e["stmt_len"]]
        assert int(e["stmt_hash"]) == py_bytes_hash(t)
        assert orc.classify(t)[0] == e["cat"]


def test_c1_bundled_corpus_summary_is_stable():
    """Config C1: the oracle over the bundled corpus's test files (committed as tests/golden/c1_testfiles.npz), summarised
    by the code that wrote the committed summary (tools/make_golden.py), reproduces every field of it."""
    import sys
    want = json.load(open(os.path.join(GOLD, "c1_summary.json")))
    assert want["n_files"] == 1779 and want["bytes"] == 10552416
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import make_golden
    fixture = os.path.join(GOLD, "c1_testfiles.npz")
    projects = bytes(np.load(fixture)["projects"]).decode().split("\n")
    files, exts, grps, _ = cu.load_fixture(fixture)
    got = make_golden.c1_summary({}, write=False, corpus=(projects, files, exts, grps))
    assert json.loads(json.dumps(got)) == want


def test_mt_harness_equals_single_thread_scan():
    """oracle/orc_mt.c (the host-cores baseline of bench.py): same records and tables as orc_scan, for any
    thread count, including more threads than files and empty files."""
    files, exts, grps = cu.fuzz_corpus(77, 300, 9000)
    files += [b""] * 40
    exts = np.concatenate([exts, np.ones(40, np.uint8)])
    grps = np.concatenate([grps, np.zeros(40, np.uint16)])
    arena, off, ln = orc.pack(files)
    want = orc.scan(arena, off, ln, exts, grps, 5, events=False)
    assert orc.lib().orc_mt_affinity_cpus() >= 1
    for threads in (1, 3, 8, 500):
        mt = orc.MtScanner(threads, max_groups=5)
        assert mt.threads == threads
        for _ in range(2):                                  # the pool is reused across calls
            got = mt.scan(arena, off, ln, exts, grps, 5)
            assert np.array_equal(got["stats"], want["stats"])
            assert np.array_equal(got["group_counts"], want["group_counts"])
            assert np.array_equal(got["global_counts"], want["global_counts"])
        mt.close()
    mt = orc.MtScanner(0)
    assert mt.threads == orc.lib().orc_mt_affinity_cpus()
    mt.close()


def test_c1_fixture_reproduces_the_committed_summary():
    """The committed C1 test files (tests/golden/c1_testfiles.npz) give the committed summary: runs on every box,
    with or without /root/reference."""
    files, exts, grps, n_groups = cu.load_fixture(os.path.join(GOLD, "c1_testfiles.npz"))
    want = json.load(open(os.path.join(GOLD, "c1_summary.json")))
    arena, off, ln = orc.pack(files)
    res = orc.scan(arena, off, ln, exts, grps, n_groups, events=False)
    st = res["stats"]
    assert len(files) == want["n_files"] and int(ln.astype(np.int64).sum()) == want["bytes"]
    assert [int(st[k].astype(np.int64).sum()) for k in ("n_lines", "n_assert", "n_headers", "n_fixture")] == \
        [want["n_lines"], want["n_assert"], want["n_headers"], want["n_fixture"]]
    assert "%016x" % int(np.bitwise_xor.reduce(st["digest"])) == want["digest_xor"]
    hz = json.load(open(os.path.join(GOLD, "ledger.json")))["C1"]
    assert hz["fixture"]["files"] == 1779 and hz["hazard_fixture"]["non_utf8"] == 1 and hz["hazard_fixture"]["crlf_files"] == 5
    hfiles, _, _, _ = cu.load_fixture(os.path.join(GOLD, "c1_hazard_files.npz"))
    assert max(len(f) for f in hfiles) == 2501857 and sum(1 for f in hfiles if f and not f.endswith(b"\n")) == 115


def test_rev_b_rules_and_golden_g1():
    """docs/SPEC.md section 4b: the later revision of the lost tool, scored against the one version-matched count golden
    (ML-Testing-v1.xlsx!DeepSpeech vs src/DeepSpeech/v0.9.3; the sheet rows ship as tests/golden/g1_deepspeech.json)."""
    assert orc.lib().orc_is_assert_line_b(b"  BOOST_CHECK_EQUAL(a, b);", 26) and not orc.is_assert_line(b"  BOOST_CHECK_EQUAL(a, b);")
    for line, ext, stmt, cat in [(b"  BOOST_CHECK_EQUAL(0xFF, x);", 2, b"BOOST_CHECK_EQUAL", "assertEqual"),
                                 (b"  BOOST_CHECK(!left.full);", 2, b"BOOST_CHECK(!left.full);", "assertFalse"),
                                 (b"  BOOST_CHECK(ref_state == test_state);", 2, b"BOOST_CHECK(ref_state == test_state);", "assertEqual"),
                                 (b"  BOOST_CHECK(base.left.full);", 2, b"BOOST_CHECK(base.left.full);", ""),
                                 (b"    assert (bufferSize > 0);", 4, b"assert (bufferSize > 0);", "assertGreater"),
                                 (b"  assert(x);", 2, b"assert", "assertTrue"),
                                 (b"  BOOST_CHECK_CLOSE(a, b, 0.1);", 2, b"BOOST_CHECK_CLOSE", ""),
                                 (b"        self.assertEqual(a, b)", 1, b"self.assertEqual", "assertEqual")]:
        arena, off, ln = orc.pack([line])
        ev = orc.scan(arena, off, ln, np.array([ext], np.uint8), np.zeros(1, np.uint16), 1, rev_b=True)["assert_events"]
        assert len(ev) == 1, line
        e = ev[0]
        assert line[e["stmt_off"]:e["stmt_off"] + e["stmt_len"]] == stmt and orc.category_name(int(e["cat"])) == cat, (line, e)
    golden = json.load(open(os.path.join(GOLD, "g1_deepspeech.json")))
    names = cu.load_fixture_names(os.path.join(GOLD, "c1_testfiles.npz"))
    files, exts, grps, n_groups = cu.load_fixture(os.path.join(GOLD, "c1_testfiles.npz"))
    keep = [i for i, n in enumerate(names) if n in golden]
    assert len(keep) == 26
    sub = [files[i] for i in keep]
    arena, off, ln = orc.pack(sub)
    ev = orc.scan(arena, off, ln, exts[keep], np.zeros(len(keep), np.uint16), 1, rev_b=True)["assert_events"]
    stm, cnt, per_file = cu.score_g1(golden, [names[i] for i in keep], sub, ev)
    assert stm == [72, 79] and cnt == [326, 427], (stm, cnt)              # canonical Rev A: 15 / 79 and 34 / 427 (ledger)
    assert per_file["DeepSpeech/v0.9.3/native_client/kenlm/util/bit_packing_test.cc"] == ([1, 1], [6, 6])   # BOOST_CHECK_EQUAL x 1, 1, 2, 2
    led = json.load(open(os.path.join(GOLD, "ledger.json")))["G1"]["rev_b"]
    assert led["sheet_statements_found"] == stm and led["assertion_count_recall"] == cnt
