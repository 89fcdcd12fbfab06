#!/usr/bin/env python3
"""Make the golden fixtures under tests/golden/ from the reference package's shipped data.

Run in the build container (needs /root/reference; the GPU box does not have it):

    python tools/make_golden.py

Outputs (all committed, all small):
  tests/golden/g4_statement_category.json   G4: (sheet, statement, category, rows) of the five Rev-A
                                            sheets of Important-files/ML-Testing-v1.xlsx
  tests/golden/g3_reduce.npz                G3: RQs/taxonomy_test2.csv reduced to integer arrays
                                            + the shipped RQ3/RQ4 table cells it must reproduce
  tests/golden/c1_summary.json              oracle totals over the bundled corpus src/ (config C1)
  tests/golden/c1_testfiles.npz             the C1 test files themselves (real bytes for the GPU box)
  tests/golden/c1_hazard_files.npz          the hazard files of SURVEY.md section 8d outside that subset
  tests/golden/g1_deepspeech.json           G1: the rows (statement -> count, category) of ML-Testing-v1.xlsx!DeepSpeech for the bundled files
  tests/golden/ledger.json                  reproduction rates of every golden (the parity ledger)

xlsx files are read with zipfile + ElementTree (no openpyxl in the image; SURVEY.md appendix A).
"""
import collections
import csv
import json
import os
import re
import sys
import zipfile
import xml.etree.ElementTree as ET

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import orc  # noqa: E402  (the oracle: this script is test infrastructure)

REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden")
NS = {"m": "http://schemas.openxmlformats.org/spreadsheetml/2006/main",
      "r": "http://schemas.openxmlformats.org/officeDocument/2006/relationships"}
REV_A = ["apollo_tests", "prefect_tests", "carma-platform_tests", "MycroftAI_tests", "donkeycar_tests"]
EXT_TAG = {"py": 1, "cc": 2, "cpp": 3, "java": 4, "c": 5, "h": 6}


def read_xlsx(path, only=None):
    z = zipfile.ZipFile(path)
    wb = ET.fromstring(z.read("xl/workbook.xml"))
    rels = {r.get("Id"): r.get("Target") for r in ET.fromstring(z.read("xl/_rels/workbook.xml.rels"))}
    ss = []
    if "xl/sharedStrings.xml" in z.namelist():
        for si in ET.fromstring(z.read("xl/sharedStrings.xml")).findall("m:si", NS):
            ss.append("".join(t.text or "" for t in si.iter("{%s}t" % NS["m"])))
    out = {}
    for sh in wb.find("m:sheets", NS):
        name = sh.get("name")
        if only and name not in only:
            continue
        t = rels[sh.get("{%s}id" % NS["r"])]
        p = "xl/" + t if not t.startswith("/") else t[1:]
        rows = []
        for row in ET.fromstring(z.read(p)).iter("{%s}row" % NS["m"]):
            cells = {}
            for c in row.findall("m:c", NS):
                m = re.match(r"([A-Z]+)(\d+)", c.get("r"))
                ci = 0
                for ch in m.group(1):
                    ci = ci * 26 + ord(ch) - 64
                ty, v = c.get("t"), c.find("m:v", NS)
                if ty == "s":
                    val = ss[int(v.text)] if v is not None else ""
                elif ty == "inlineStr":
                    val = "".join(t.text or "" for t in c.iter("{%s}t" % NS["m"]))
                else:
                    val = v.text if v is not None else ""
                cells[ci - 1] = val
            rows.append((int(row.get("r")), [cells.get(i, "") for i in range(max(cells) + 1)] if cells else []))
        out[name] = rows
    return out


def golden_g4(v1, ledger):
    pairs = collections.Counter()
    per_sheet = {}
    for sh in REV_A:
        hit = n = 0
        for _, r in v1[sh][1:]:
            if len(r) < 7 or r[4] == "[]":
                continue
            n += 1
            pairs[(sh, r[4], r[6])] += 1
            if orc.category_string(r[4].encode("utf-8")) == r[6]:
                hit += 1
        per_sheet[sh] = [hit, n]
    rows = [{"sheet": s, "statement": t, "category": c, "rows": k} for (s, t, c), k in sorted(pairs.items())]
    misses = [r for r in rows if orc.category_string(r["statement"].encode("utf-8")) != r["category"]]
    json.dump(rows, open(os.path.join(OUT, "g4_statement_category.json"), "w"), indent=0, ensure_ascii=True)
    tot = [sum(v[0] for v in per_sheet.values()), sum(v[1] for v in per_sheet.values())]
    # S4 truncation rule: no statement keeps a '(' and none has surrounding blanks
    trunc_ok = sum(k for (s, t, c), k in pairs.items() if "(" not in t and t == t.strip())
    ledger["G4"] = {"source": "Important-files/ML-Testing-v1.xlsx, sheets " + ", ".join(REV_A),
                    "category_rule_rows": tot, "per_sheet": per_sheet,
                    "truncation_rule_rows": [trunc_ok, tot[1]],
                    "misses": [{"statement": m["statement"], "sheet_says": m["category"],
                                "oracle_says": orc.category_string(m["statement"].encode("utf-8")),
                                "rows": m["rows"]} for m in misses]}
    print("G4", tot, "misses", len(misses))


def oracle_rows(data, ext):
    """(method, statement) -> count for one file, via the oracle's line-level functions."""
    out = collections.Counter()
    cur = b"xxxx"
    pos = 0
    while pos < len(data):
        e = data.find(b"\n", pos)
        if e < 0:
            e = len(data)
        line = data[pos:e]
        if orc.header_kind(ext, line):
            cur = orc.method_string(ext, line)
        if orc.is_assert_line(line):
            out[(cur, orc.statement(line))] += 1
        pos = e + 1
    return out


def ledger_headers(v1, ledger):
    """S3 header rule on the apollo_tests files that exist in the bundled (version-skewed) snapshot."""
    root = os.path.join(REF, "src/apollo/v6.0.0")
    by = collections.defaultdict(collections.Counter)
    for _, r in v1["apollo_tests"][1:]:
        if len(r) >= 7:
            by[r[0]][(r[3].encode(), r[4].encode())] += int(float(r[5]))
    hit = tot = files_exact = files = 0
    for f, want in by.items():
        p = os.path.join(root, f)
        if not os.path.exists(p):
            continue
        files += 1
        got = oracle_rows(open(p, "rb").read(), EXT_TAG.get(f.rsplit(".", 1)[-1], 0))
        ok = True
        for k, v in want.items():
            tot += 1
            if got.get(k) == v:
                hit += 1
            else:
                ok = False
        files_exact += ok and set(got) == set(want)
    ledger["S3_apollo"] = {"source": "ML-Testing-v1.xlsx!apollo_tests vs src/apollo/v6.0.0 (version-skewed)",
                           "files_in_bundle": [files, len(by)], "rows_exact": [hit, tot],
                           "files_exact": [files_exact, files]}
    print("S3 apollo", hit, tot, files_exact, files)


def ledger_g1(v1, ledger):
    root = os.path.join(REF, "src/DeepSpeech/v0.9.3")
    by = collections.defaultdict(collections.Counter)
    for _, r in v1["DeepSpeech"][1:]:
        if len(r) >= 7:
            by[r[0]][r[4]] += int(float(r[5]))
    files = stm_hit = stm_tot = cnt_hit = cnt_tot = 0
    for f, want in by.items():
        p = os.path.join(root, f)
        if not os.path.exists(p):
            continue
        files += 1
        data = open(p, "rb").read()
        ext = EXT_TAG.get(f.rsplit(".", 1)[-1], 0)
        got_full = collections.Counter()
        got_trunc = collections.Counter()
        pos = 0
        while pos < len(data):
            e = data.find(b"\n", pos)
            e = len(data) if e < 0 else e
            line = data[pos:e]
            if orc.is_assert_line(line):
                got_trunc[orc.statement(line).decode("latin-1")] += 1
                got_full[line.decode("latin-1").strip(" \t\r\x0b\x0c")] += 1
            pos = e + 1
        for st, c in want.items():
            stm_tot += 1
            cnt_tot += c
            g = got_trunc.get(st) or got_full.get(st)
            if g:
                stm_hit += 1
                cnt_hit += min(c, g)
    # ---- the same sheet scored with the Rev-B mode of the oracle (docs/SPEC.md section 4b), and the sheet rows of the bundled
    #      files as a fixture (tests/golden/g1_deepspeech.json) so that the GPU box can score the CUDA path against G1
    fixture, b_stm = {}, [0, 0]
    b_cnt, b_cat = [0, 0], [0, 0]
    cats = collections.defaultdict(dict)
    for _, r in v1["DeepSpeech"][1:]:
        if len(r) >= 7:
            cats[r[0]][r[4]] = r[6]
    per_file = {}
    for f, want in sorted(by.items()):
        p = os.path.join(root, f)
        if not os.path.exists(p):
            continue
        data = open(p, "rb").read()
        ext = EXT_TAG.get(f.rsplit(".", 1)[-1], 0)
        arena, off, ln = orc.pack([data])
        res = orc.scan(arena, off, ln, np.array([ext], np.uint8), np.zeros(1, np.uint16), 1, rev_b=True)
        got, gcat = collections.Counter(), {}
        for e in res["assert_events"]:
            st = data[e["stmt_off"]:e["stmt_off"] + e["stmt_len"]].decode("latin-1")
            got[st] += 1
            gcat[st] = orc.category_name(int(e["cat"])) if e["cat"] != 127 else data[e["ident_off"]:e["ident_off"] + e["ident_len"]].decode("latin-1")
        fixture["DeepSpeech/v0.9.3/" + f] = {st: [c, cats[f][st]] for st, c in want.items()}
        fs = fc = 0
        for st, c in want.items():
            b_stm[1] += 1
            b_cnt[1] += c
            if got.get(st):
                b_stm[0] += 1
                b_cnt[0] += min(c, got[st])
                fs += 1
                fc += min(c, got[st])
                b_cat[1] += 1
                b_cat[0] += gcat[st] == cats[f][st]
        per_file[f] = {"statements": [fs, len(want)], "counts": [fc, sum(want.values())]}
    json.dump(fixture, open(os.path.join(OUT, "g1_deepspeech.json"), "w"), indent=0, sort_keys=True)
    assert per_file["native_client/kenlm/util/bit_packing_test.cc"] == {"statements": [1, 1], "counts": [6, 6]}
    ledger["G1"] = {"rev_b": {"rule": "docs/SPEC.md section 4b", "sheet_statements_found": b_stm, "assertion_count_recall": b_cnt,
                              "category_agreement_on_found_statements": b_cat, "per_file": per_file},
                    "source": "ML-Testing-v1.xlsx!DeepSpeech (Rev-B sheet) vs src/DeepSpeech/v0.9.3",
                    "files_in_bundle": [files, len(by)],
                    "sheet_statements_found_as_truncated_or_full_line": [stm_hit, stm_tot],
                    "assertion_count_recall": [cnt_hit, cnt_tot],
                    "note": "the two lists above are canonical Rev A scored on the Rev-B sheet; Rev B also triggers on _CHECK / TESTEQUAL / FAIL"}
    print("G1 rev A", stm_hit, stm_tot, cnt_hit, cnt_tot, "| rev B", b_stm, b_cnt, "category", b_cat)


# Error_Type values merged into one strategy row.  Not written down anywhere in the package: recovered by exhaustive
# search over the 2^20 value subsets against the nine per-repository cells of tests_strategy_rq32.csv - each of the
# three sets is the unique (runtime_error: minimal of two, the other adds the one-case `ConfigError`) exact solution.
RUNTIME = ("RuntimeError", "Exception", "NotImplementedError", "StopIteration", "TimeOut", "Timeout", "TimeoutError",
           "Warning", "nullptr")
STRATEGY = [  # (row name in tests_strategy_rq32.csv, column, value or tuple of values)
    ("status_analysis", "status_test", "1"), ("value_error", "Error_Type", "ValueError"),
    ("runtime_error", "Error_Type", RUNTIME), ("memory_error", "Error_Type", "MemoryError"),
    ("type_error", "Error_Type", "TypeError"), ("import_error", "Error_Type", "ImportError"),
    ("key_error", "Error_Type", "KeyError"), ("AssertionError", "Error_Type", ("AssertionError", "SyntaxError")),
    ("FileError", "Error_Type", ("FileError", "SchemaError")), ("NotImplementedError", "Error_Type", "NotImplementedError"),
    ("negative_test", "negative_test", "1"), ("logical_condition", "logical_statement", "1"),
    ("Null_pointer", "null_pointer", "1"), ("value_range", "value_range", "1"),
    ("absolute_relative_tolerence", "Approximation_Type", "absolute_relative_tolerence"),
    ("error_bounding", "Approximation_Type", "error_bounding"),
    ("rounding_tolence", "Approximation_Type", "rounding_tolence"),
    ("instance_check", "checks_type", "instance_check"), ("sub_set_checks", "checks_type", "sub_set_checks")]
METHODS = [  # (row name in tests_methods_v2.csv, taxonomy column)
    ("regression", "regression"), ("integration", "Integration"), ("end_to_end", "end_to_end"),
    ("sanity", "sanity"), ("mock_test", "mock_test"), ("periodic_validation", "periodic_validation"),
    ("example_test", "example_test"), ("static_inspection", "static_inspection_test"),
    ("robustness_test", "roboustness"), ("experimental", "Experimental_benchmark_test"),
    ("api_test", "API"), ("threat", "ThreadTest"), ("blob", "blob_performance")]


# RQ3 property table (tests_prop_rq3.csv): property -> Data / Model labels.  17 of the 21 sets are exact solutions of a
# search against the nine shipped per-repository cells; Consistency, Features Importance, Concurrency and Anomaly are
# not recoverable from taxonomy_test2.csv (their cells need labels this revision of the CSV does not carry).
PROPERTIES = [
    ("Consistency", ("Consistency",)), ("Data Distribution", ("Distribution",)),
    ("Data Validity", ("Validity", "Data Error", "Data Error and Validity")), ("Completeness", ("Completeness",)),
    ("Correctness", ("Correctness", "Accuracy & Precision", "Statistical Evidence/ explainability")),
    ("Robustness", ("Robustness",)), ("Efficiency", ("Time behaviour", "Resource Usage", "Training Efficiency")),
    ("Data Relation", ("Relation & Association", "Closeness", "Missing Data", "Data Differencing", "Data Quality")),
    ("Scalability", ("Scalability",)), ("Features Importance", ("Feature Importance",)),
    ("Data Restoration and Recoverability", ("Recoverability", "Data Restoration")),
    ("Concurrency and Parallelism", ("Parallel Processing", "parallel")), ("Uncertainty", ("uncertainty",)),
    ("Anomaly", ("Anomaly",)), ("Data Migration Loss and Corruption", ("Data Loss",)),
    ("Bias and Fairness", ("Model Bias",)), ("Security and Privacy", ("Security", "Data Encapsulation")),
    ("Data Uniqueness", ("Uniqueness",)), ("Data Timeliness", ("Timeliness",)),
    ("Data Integration Integrity", ("Validate data integration and integrity",)),
    ("Compatibility and Portability", ("Compatibility",))]


# RQ3 strategy x property table (RQs/RQ3/tests_correlate_rq3.csv): 20 strategy rows, 21 property columns, one cell =
# "repo:(p%), " over the nine repositories, p = 100 * distinct cases with BOTH flags / cases of the repository, rounded
# to 2 decimals and printed as a Python float ("0.0", "1.22", "12.2"); a cell with no case at all is the string "0".
# The row predicates are single taxonomy values (unlike tests_strategy_rq32.csv, which merges Error_Type values):
# `decision` is logical_statement, `logical_condition` is logical_expression (recovered against the shipped cells).
CORRELATE_ROWS = [  # (row name in tests_correlate_rq3.csv, column, value)
    ("rounding_tolence", "Approximation_Type", "rounding_tolence"), ("instance_check", "checks_type", "instance_check"),
    ("MemoryError", "Error_Type", "MemoryError"), ("negative_test", "negative_test", "1"),
    ("status_analysis", "status_test", "1"), ("value_range_analysis", "value_range", "1"),
    ("sub_set_checks", "checks_type", "sub_set_checks"), ("ValueError", "Error_Type", "ValueError"),
    ("decision", "logical_statement", "1"), ("error_bounding", "Approximation_Type", "error_bounding"),
    ("Null_pointer", "null_pointer", "1"), ("boundary", "boundary", "1"),
    ("absolute_relative_tolerence", "Approximation_Type", "absolute_relative_tolerence"),
    ("ImportError", "Error_Type", "ImportError"), ("pseaudo_oracle", "Pseaudo_Oracle", "1"),
    ("RuntimeError", "Error_Type", "RuntimeError"), ("logical_condition", "logical_expression", "1"),
    ("TypeError", "Error_Type", "TypeError"), ("KeyError", "Error_Type", "KeyError"),
    ("NotImplementedError", "Error_Type", "NotImplementedError")]
CORRELATE_COLS = [  # (column name in tests_correlate_rq3.csv, name in PROPERTIES)
    ("Distribution", "Data Distribution"), ("Validity", "Data Validity"), ("Consistency", "Consistency"),
    ("Completeness", "Completeness"), ("Correctness", "Correctness"), ("Robustness", "Robustness"),
    ("Efficiency", "Efficiency"), ("Relation", "Data Relation"), ("Scalability", "Scalability"),
    ("Feature Importance", "Features Importance"), ("Restoration", "Data Restoration and Recoverability"),
    ("Concurrency", "Concurrency and Parallelism"), ("uncertainty", "Uncertainty"), ("Anomaly", "Anomaly"),
    ("Data Loss", "Data Migration Loss and Corruption"), ("Bias", "Bias and Fairness"),
    ("Security", "Security and Privacy"), ("Uniqueness", "Data Uniqueness"), ("Timeliness", "Data Timeliness"),
    ("integration", "Data Integration Integrity"), ("Compatibility", "Compatibility and Portability")]
CORRELATE_REPOS = ["auto_sklearn", "google_automl", "tpot", "autokeras", "Nupic", "Apollo", "nni", "Ray", "DeepSpeech2"]


def correlate_cell(distinct, cases, names):
    """One cell of tests_correlate_rq3.csv from the distinct-case counts of the nine repositories."""
    if not any(distinct):
        return "0"
    return "".join("%s:(%s%%), " % (n, repr(round(100.0 * int(d) / int(c), 2))) for n, d, c in zip(names, distinct, cases))


def fmt4(x):
    s = ("%.4f" % x).rstrip("0").rstrip(".")
    return s if s else "0"


def rq3_cell(distinct, cases):
    """Shipped cells are rounded twice: 26/142 -> 18.3099 -> /1.1 -> 16.6454 (tests_strategy_rq32.csv:3, tpot)."""
    return fmt4(round(round(100.0 * distinct / cases, 4) / 1.1, 4))


def golden_g3(ledger):
    rows = list(csv.DictReader(open(os.path.join(REF, "RQs/taxonomy_test2.csv"), newline="", encoding="utf-8")))
    repos = ["autokeras", "auto_sklearn", "tpot", "Ray", "DeepSpeech2", "google_automl", "nni", "Apollo", "Nupic"]
    rid = {r: i for i, r in enumerate(repos)}
    cases = sorted({r["Cases"] for r in rows}, key=lambda s: (len(s), s))
    cid = {c: i for i, c in enumerate(cases)}
    names = [s[0] for s in STRATEGY] + ["m:" + m[0] for m in METHODS] + ["p:" + q[0] for q in PROPERTIES]
    flags = np.zeros((len(rows), len(names)), np.uint8)
    for i, r in enumerate(rows):
        for j, (name, col, val) in enumerate(STRATEGY):
            flags[i, j] = r[col].strip() in (val if isinstance(val, tuple) else (val,))
            if name == "logical_condition":
                flags[i, j] |= r["logical_expression"].strip() == "1"
        for j, (_, col) in enumerate(METHODS):
            flags[i, len(STRATEGY) + j] = r[col].strip() not in ("", "0")
        for j, (_, labels) in enumerate(PROPERTIES):
            flags[i, len(STRATEGY) + len(METHODS) + j] = (r["Data"].strip() in labels) or (r["Model"].strip() in labels)
    repo = np.array([rid[r["Repo"]] for r in rows], np.int32)
    case = np.array([cid[r["Cases"]] for r in rows], np.int32)
    out, cpr = orc.reduce(flags, repo, case, len(repos), len(cases))
    # shipped tables
    t = list(csv.reader(open(os.path.join(REF, "RQs/RQ3/tests_strategy_rq32.csv"), newline="")))
    assert t[0][1:10] == repos
    want3 = {r[0]: r[1:10] for r in t[1:] if r and r[0]}
    cell_ok = np.zeros((len(STRATEGY), len(repos)), np.uint8)
    want_cells = []
    for j, (name, _, _) in enumerate(STRATEGY):
        want_cells.append(want3[name])
        for k in range(len(repos)):
            mine = rq3_cell(out[j, k], cpr[k])
            cell_ok[j, k] = mine == want3[name][k]
    t4 = list(csv.DictReader(open(os.path.join(REF, "RQs/RQ4/tests_methods_v2.csv"), newline="")))
    want4 = {r["Test_methods"]: int(r["total_cases"]) for r in t4}
    m_ok = []
    # RQ4: distinct cases over all repos = sum over repos (a case belongs to one repo)
    for j, (name, _) in enumerate(METHODS):
        m_ok.append(int(out[len(STRATEGY) + j].sum()) == want4[name])
    # the columns `tosem-scan reduce` reads, as a compact fixture for the CLI's own golden test (tests/test_cli.py)
    import gzip
    keep = ["Cases", "Repo", "Data", "Model"] + sorted({c for _, c, _ in STRATEGY} | {c for _, c, _ in CORRELATE_ROWS} | {c for _, c in METHODS})
    import io
    txt = io.StringIO(newline="")
    w = csv.writer(txt, lineterminator="\r\n")
    w.writerow(keep)
    for r in rows:
        w.writerow([r[c] for c in keep])
    with open(os.path.join(OUT, "taxonomy_min.csv.gz"), "wb") as raw:      # mtime 0, no file name: the bytes do not
        with gzip.GzipFile(filename="", mode="wb", fileobj=raw, compresslevel=9, mtime=0) as f:   # depend on when it is made
            f.write(txt.getvalue().encode("utf-8"))
    # RQ3 property table: rows = repos (shipped order), cells = 100 * distinct / 216
    tp = list(csv.reader(open(os.path.join(REF, "RQs/RQ3/tests_prop_rq3.csv"), newline="")))
    assert tp[0][1:] == [q[0] for q in PROPERTIES]
    prop_rows = [r for r in tp[1:10]]
    denom = int(cpr[rid["Apollo"]])           # 216: the shipped table divides every repository by Apollo's case count
    prop_ok = np.zeros((len(PROPERTIES), len(repos)), np.uint8)
    want_prop = [["" for _ in repos] for _ in PROPERTIES]
    p0 = len(STRATEGY) + len(METHODS)
    for r in prop_rows:
        k = rid[r[0]]
        for j in range(len(PROPERTIES)):
            want_prop[j][k] = r[1 + j]
            prop_ok[j, k] = fmt4(round(100.0 * out[p0 + j, k] / denom, 4)) == r[1 + j]
    # RQ3 strategy x property table: 20 x 21 combined flags through the same reduction
    labels_of = dict(PROPERTIES)
    cflags = np.zeros((len(rows), len(CORRELATE_ROWS) * len(CORRELATE_COLS)), np.uint8)
    for i, r in enumerate(rows):
        pr = [(r["Data"].strip() in labels_of[q]) or (r["Model"].strip() in labels_of[q]) for _, q in CORRELATE_COLS]
        for j, (_, col, val) in enumerate(CORRELATE_ROWS):
            if r[col].strip() == val:
                cflags[i, j * len(CORRELATE_COLS):(j + 1) * len(CORRELATE_COLS)] = pr
    cout, _ = orc.reduce(cflags, repo, case, len(repos), len(cases))
    tc = list(csv.reader(open(os.path.join(REF, "RQs/RQ3/tests_correlate_rq3.csv"), newline="")))
    assert tc[0][1:] == [c for c, _ in CORRELATE_COLS] and [r[0] for r in tc[1:]] == [r[0] for r in CORRELATE_ROWS]
    order = [rid[n] for n in CORRELATE_REPOS]
    corr_ok = np.zeros((len(CORRELATE_ROWS), len(CORRELATE_COLS)), np.uint8)
    want_corr = [r[1:] for r in tc[1:]]
    for j in range(len(CORRELATE_ROWS)):
        for q in range(len(CORRELATE_COLS)):
            d = cout[j * len(CORRELATE_COLS) + q]
            corr_ok[j, q] = correlate_cell([d[k] for k in order], [cpr[k] for k in order], CORRELATE_REPOS) == want_corr[j][q]
    # the same counts in the two other shipped layouts: LaTeX cells that list the non-zero repositories only
    # (tests_correlate_rq4.csv), and the distinct cases of all repositories together (tests_combined_correlate_rq3.csv)
    ttex = list(csv.reader(open(os.path.join(REF, "RQs/RQ3/tests_correlate_rq4.csv"), newline="")))
    tcnt = list(csv.reader(open(os.path.join(REF, "RQs/RQ3/tests_combined_correlate_rq3.csv"), newline="", encoding="utf-8-sig")))
    assert ttex[0] == tc[0] and tcnt[0] == tc[0] and [r[0] for r in ttex[1:]] == [r[0] for r in tc[1:]] == [r[0] for r in tcnt[1:]]
    tex_ok = np.zeros_like(corr_ok)
    cnt_ok = np.zeros_like(corr_ok)
    for j in range(len(CORRELATE_ROWS)):
        for q in range(len(CORRELATE_COLS)):
            d = cout[j * len(CORRELATE_COLS) + q]
            tex = "".join("$%s:%s\\%%$, " % (n, repr(round(100.0 * int(d[k]) / int(cpr[k]), 2))) for n, k in zip(CORRELATE_REPOS, order) if d[k]) or "0"
            tex_ok[j, q] = tex == ttex[1 + j][1 + q]
            cnt_ok[j, q] = str(int(d.sum())) == tcnt[1 + j][1 + q]
    # four more one-row tables in the correlate layout, for the MERGED strategy rows of tests_strategy_rq32.csv
    # (tests_correlate_{FileError,RuntimeError,assertion,logical}.csv): the same value sets as STRATEGY above
    merged_rows = [("FileError", "FileError", "FileError"), ("RuntimeError", "RuntimeError", "runtime_error"),
                   ("AssertionError", "assertion", "AssertionError"), ("logical", "logical", "logical_condition")]   # (row name, file suffix, STRATEGY row)
    sidx = {name: j for j, (name, _, _) in enumerate(STRATEGY)}
    mflags = np.zeros((len(rows), len(merged_rows) * len(CORRELATE_COLS)), np.uint8)
    for i, r in enumerate(rows):
        pr = [(r["Data"].strip() in labels_of[q]) or (r["Model"].strip() in labels_of[q]) for _, q in CORRELATE_COLS]
        for j, (_, _, srow) in enumerate(merged_rows):
            if flags[i, sidx[srow]]:
                mflags[i, j * len(CORRELATE_COLS):(j + 1) * len(CORRELATE_COLS)] = pr
    mout, _ = orc.reduce(mflags, repo, case, len(repos), len(cases))
    merged_ok = np.zeros((len(merged_rows), len(CORRELATE_COLS)), np.uint8)
    want_merged = []
    for j, (rname, suffix, _) in enumerate(merged_rows):
        tm = list(csv.reader(open(os.path.join(REF, "RQs/RQ3/tests_correlate_%s.csv" % suffix), newline="")))
        assert tm[0] == tc[0] and len(tm) == 2 and tm[1][0] == rname, (suffix, tm[1][0])
        want_merged.append(tm[1][1:])
        for q in range(len(CORRELATE_COLS)):
            d = mout[j * len(CORRELATE_COLS) + q]
            merged_ok[j, q] = correlate_cell([d[k] for k in order], [cpr[k] for k in order], CORRELATE_REPOS) == tm[1][1 + q]
    np.savez_compressed(os.path.join(OUT, "g3_reduce.npz"), flags=flags, repo=repo, case_id=case,
                        want_property_cells=np.array(want_prop), property_cell_reproduces=prop_ok,
                        flag_names=np.array(names), repo_names=np.array(repos),
                        want_strategy_cells=np.array(want_cells), strategy_cell_reproduces=cell_ok,
                        want_method_total_cases=np.array([want4[m[0]] for m in METHODS], np.int64),
                        method_reproduces=np.array(m_ok, np.uint8),
                        oracle_distinct=out, oracle_cases_per_repo=cpr,
                        want_correlate_cells=np.array(want_corr), correlate_cell_reproduces=corr_ok,
                        correlate_row_names=np.array([r[0] for r in CORRELATE_ROWS]),
                        correlate_col_names=np.array([c for c, _ in CORRELATE_COLS]),
                        correlate_row_column=np.array([r[1] for r in CORRELATE_ROWS]),
                        correlate_row_value=np.array([r[2] for r in CORRELATE_ROWS]),
                        correlate_col_labels=np.array(["|".join(labels_of[q]) for _, q in CORRELATE_COLS]),
                        correlate_repo_order=np.array(CORRELATE_REPOS), oracle_correlate_distinct=cout,
                        want_correlate_tex_cells=np.array([r[1:] for r in ttex[1:]]), correlate_tex_cell_reproduces=tex_ok,
                        want_correlate_count_cells=np.array([r[1:] for r in tcnt[1:]]), correlate_count_cell_reproduces=cnt_ok,
                        merged_row_names=np.array([m[0] for m in merged_rows]), merged_strategy_rows=np.array([m[2] for m in merged_rows]),
                        want_merged_cells=np.array(want_merged), merged_cell_reproduces=merged_ok, oracle_merged_distinct=mout)
    ledger["G3"] = {"source": "RQs/taxonomy_test2.csv -> RQs/RQ3/tests_strategy_rq32.csv, RQs/RQ4/tests_methods_v2.csv",
                    "rows": len(rows), "cases": len(cases), "cases_per_repo": dict(zip(repos, map(int, cpr))),
                    "strategy_cells_bit_identical": [int(cell_ok.sum()), int(cell_ok.size)],
                    "rq4_method_counts_identical": [int(sum(m_ok)), len(m_ok)],
                    "property_cells_bit_identical": [int(prop_ok.sum()), int(prop_ok.size)],
                    "property_columns_fully_identical": [int((prop_ok.sum(axis=1) == len(repos)).sum()), len(PROPERTIES)],
                    "correlate_cells_bit_identical": [int(corr_ok.sum()), int(corr_ok.size)],
                    "correlate_rows_fully_identical": [int((corr_ok.sum(axis=1) == len(CORRELATE_COLS)).sum()), len(CORRELATE_ROWS)],
                    "correlate_tex_cells_bit_identical (tests_correlate_rq4.csv)": [int(tex_ok.sum()), int(tex_ok.size)],
                    "correlate_count_cells_identical (tests_combined_correlate_rq3.csv)": [int(cnt_ok.sum()), int(cnt_ok.size)],
                    "merged_row_cells_bit_identical (tests_correlate_{FileError,RuntimeError,assertion,logical}.csv)":
                        {m[0]: [int(merged_ok[j].sum()), len(CORRELATE_COLS)] for j, m in enumerate(merged_rows)},
                    "rq4_mismatches": {m[0]: [int(out[len(STRATEGY) + j].sum()), want4[m[0]]]
                                       for j, m in enumerate(METHODS) if not m_ok[j]}}
    print("G3 cells", int(cell_ok.sum()), cell_ok.size, "rq4", sum(m_ok), len(m_ok), "property cells", int(prop_ok.sum()), prop_ok.size,
          "correlate cells", int(corr_ok.sum()), corr_ok.size)


def c1_collect():
    """The test files of the bundled corpus with a scannable extension (S0 + S1), in walk order."""
    root = os.path.join(REF, "src")
    projects = sorted(os.listdir(root))
    projects = [p for p in projects if os.path.isdir(os.path.join(root, p))]
    files, ext, grp, names = [], [], [], []
    for g, proj in enumerate(projects):
        base = os.path.join(root, proj)
        vers = sorted(os.listdir(base))
        vroot = os.path.join(base, vers[0]) if len(vers) == 1 and os.path.isdir(os.path.join(base, vers[0])) else base
        for dp, dn, fn in os.walk(vroot):
            dn.sort()
            for f in sorted(fn):
                e = f.rsplit(".", 1)[-1] if "." in f else ""
                rel = os.path.relpath(os.path.join(dp, f), vroot)
                if e not in EXT_TAG or "test" not in rel.lower():
                    continue
                files.append(open(os.path.join(dp, f), "rb").read())
                ext.append(EXT_TAG[e])
                grp.append(g)
                names.append(proj + "/" + rel)
    return projects, files, ext, grp, names


def c1_fixture():
    """tests/golden/c1_testfiles.npz: the C1 test files themselves (1 779 files, 10.55 MB of the study's corpus),
    so that the GPU box - which has no /root/reference - can put real bytes through the CUDA path.  Deflated."""
    projects, files, ext, grp, names = c1_collect()
    blob = np.frombuffer(b"".join(files), np.uint8)
    np.savez_compressed(os.path.join(OUT, "c1_testfiles.npz"), blob=blob, size=np.array([len(f) for f in files], np.int32),
                        ext=np.array(ext, np.uint8), grp=np.array(grp, np.uint16),
                        names=np.frombuffer("\n".join(names).encode(), np.uint8),
                        projects=np.frombuffer("\n".join(projects).encode(), np.uint8))
    hz = {"files": len(files), "bytes": int(blob.size), "empty": sum(1 for f in files if not f),
          "crlf_files": sum(1 for f in files if b"\r\n" in f), "no_trailing_newline": sum(1 for f in files if f and not f.endswith(b"\n")),
          "with_bytes_over_127": sum(1 for f in files if any(b > 127 for b in f)), "largest": max(len(f) for f in files),
          "longest_line": max(max((len(l) for l in f.split(b"\n")), default=0) for f in files)}
    print("C1 fixture", hz)
    return hz


def c1_hazards():
    """tests/golden/c1_hazard_files.npz: the hazard files SURVEY.md section 8d lists for config C1 that lie outside the
    test-file subset: the one non-UTF-8 file, every CRLF file, the 2.5 MB file with the 2 061-byte lines, and every
    scannable file without a trailing newline."""
    root = os.path.join(REF, "src")
    picked = []
    for dp, dn, fn in os.walk(root):
        dn.sort()
        for f in sorted(fn):
            e = f.rsplit(".", 1)[-1] if "." in f else ""
            if e not in EXT_TAG:
                continue
            b = open(os.path.join(dp, f), "rb").read()
            try:
                b.decode("utf-8")
                utf8 = True
            except UnicodeDecodeError:
                utf8 = False
            if (not utf8) or b"\r\n" in b or len(b) > 2500000 or (b and not b.endswith(b"\n")):
                picked.append((os.path.relpath(os.path.join(dp, f), root), b, EXT_TAG[e]))
    blob = np.frombuffer(b"".join(b for _, b, _ in picked), np.uint8)
    np.savez_compressed(os.path.join(OUT, "c1_hazard_files.npz"), blob=blob, size=np.array([len(b) for _, b, _ in picked], np.int32),
                        ext=np.array([e for _, _, e in picked], np.uint8), grp=np.zeros(len(picked), np.uint16),
                        names=np.frombuffer("\n".join(n for n, _, _ in picked).encode(), np.uint8))
    hz = {"files": len(picked), "bytes": int(blob.size), "non_utf8": sum(1 for _, b, _ in picked if not _is_utf8(b)),
          "crlf_files": sum(1 for _, b, _ in picked if b"\r\n" in b),
          "no_trailing_newline": sum(1 for _, b, _ in picked if b and not b.endswith(b"\n")),
          "largest": max(len(b) for _, b, _ in picked),
          "longest_line": max(max((len(l) for l in b.split(b"\n")), default=0) for _, b, _ in picked)}
    print("C1 hazards", hz)
    return hz


def _is_utf8(b):
    try:
        b.decode("utf-8")
        return True
    except UnicodeDecodeError:
        return False


def c1_summary(ledger, write=True, corpus=None):
    """Config C1: the oracle over the bundled corpus (test files with a scannable extension).  corpus = (projects,
    files, ext, grp) of those files from elsewhere: the tests pass tests/golden/c1_testfiles.npz."""
    projects, files, ext, grp = corpus or c1_collect()[:4]
    arena, off, length = orc.pack(files)
    res = orc.scan(arena, off, length, np.array(ext, np.uint8), np.array(grp, np.uint16), len(projects), events=False)
    st = res["stats"]
    summ = {"projects": projects, "n_files": len(files), "bytes": int(length.astype(np.int64).sum()),
            "n_lines": int(st["n_lines"].astype(np.int64).sum()),
            "n_assert": int(st["n_assert"].astype(np.int64).sum()),
            "n_headers": int(st["n_headers"].astype(np.int64).sum()),
            "n_fixture": int(st["n_fixture"].astype(np.int64).sum()),
            "digest_xor": "%016x" % int(np.bitwise_xor.reduce(st["digest"])),
            "global_counts": {orc.category_name(i) or "''": int(c) for i, c in enumerate(res["global_counts"]) if c},
            "per_project_assert": {p: int(res["group_counts"][g].sum()) for g, p in enumerate(projects)}}
    if not write:
        return summ
    json.dump(summ, open(os.path.join(OUT, "c1_summary.json"), "w"), indent=1)
    ledger["C1"] = {"source": "src/** (test-path files with extension py/cc/cpp/java/c/h)",
                    "n_files": summ["n_files"], "bytes": summ["bytes"], "n_lines": summ["n_lines"],
                    "n_assert": summ["n_assert"], "n_headers": summ["n_headers"],
                    "survey_says": {"n_files": 1779, "bytes": 10552416, "n_lines": 296147,
                                    "n_headers": 6190, "n_assert": 26046}}
    print("C1", summ["n_files"], summ["bytes"], summ["n_lines"], summ["n_assert"], summ["n_headers"])


ANNOTATION = re.compile(r"^(compare|approximate|approximation|error-handling|value-range( nested)?|logical statement|else:|check)\s+", re.I)


def ledger_g2(ledger):
    """Golden G2 (body statements, SPEC section 10): recall of the verbatim sheet rows of ML-Analysis-v4.xlsx among the
    oracle's statements of the FileID-mapped source file (SURVEY.md appendix A for the FileID -> path joins)."""
    def idmap_xlsx(path, ci, cp):
        sh = list(read_xlsx(path).values())[0]
        out = {}
        for _, row in sh[1:]:
            if len(row) > max(ci, cp) and row[ci]:
                try:
                    out[int(float(row[ci]))] = row[cp]
                except ValueError:
                    pass
        return out

    def idmap_csv(path):
        out = {}
        for row in csv.DictReader(open(path, newline="", encoding="utf-8")):
            try:
                out[int(float(row["Id"]))] = row["FileName"]
            except (ValueError, KeyError):
                pass
        return out
    lab = os.path.join(REF, "selection/completed-labels")
    subjects = {"Apollo": (idmap_xlsx(os.path.join(lab, "Release-Meta-Apollo_2.xlsx"), 0, 1), "src/apollo/v6.0.0"),
                "DeepSpeech2": (idmap_xlsx(os.path.join(lab, "Release-Meta-Deepspeech_2.xlsx"), 1, 2), "src/DeepSpeech/v0.9.3"),
                "Nupic": (idmap_xlsx(os.path.join(lab, "Release-Meta-nupic_22.xlsx"), 1, 2), "src/nupic/1.0.5"),
                "autokeras": (idmap_csv(os.path.join(lab, "Release-Meta-autokeras.csv")), "src/autokeras/1.0.12")}
    v4 = read_xlsx(os.path.join(REF, "Important-files/ML-Analysis-v4.xlsx"), only=set(subjects))

    def norm(t):
        return re.sub(r"\s+", " ", t).strip()
    out = {}
    for name, (fid, root) in subjects.items():
        by = collections.defaultdict(list)
        for _, r in v4[name][1:]:
            if len(r) >= 5 and r[4]:
                try:
                    by[int(float(r[4]))].append(r[1])
                except ValueError:
                    pass
        hit = tot = files = 0
        for f, texts in by.items():
            p = fid.get(f)
            if not p or not os.path.exists(os.path.join(REF, root, p)):
                continue
            files += 1
            data = open(os.path.join(REF, root, p), "rb").read()
            text = data.decode("utf-8", "replace")
            have = {norm(x.decode("utf-8", "replace")) for x in orc.statement_texts(data)}
            for t in texts:
                t = norm(t)
                if not t:
                    continue
                tot += 1
                if t in have or norm(ANNOTATION.sub("", t)) in have:
                    hit += 1
                elif re.match(r"^[A-Za-z_0-9(), .:]+$", t) and len(t) < 80 and (t in text or t.split("(")[0] in text):
                    hit += 1                                   # case-name rows (GetAllCorners, TEST_CASE(Query), testNoShift)
        out[name] = {"files_in_bundle": files, "rows_recalled": [hit, tot]}
        print("G2", name, hit, tot)
    ledger["G2"] = {"source": "Important-files/ML-Analysis-v4.xlsx!{Apollo,DeepSpeech2,Nupic,autokeras} vs the bundled sources",
                    "rule": "docs/SPEC.md section 10 (lines joined while the parentheses are open)", "subjects": out,
                    "note": "recall of verbatim rows; the residue is labeller paraphrase and version skew (SURVEY.md section 8c)"}


def main():
    if "--check-c1" in sys.argv:   # recompute config C1 and compare with the committed summary
        want = json.load(open(os.path.join(OUT, "c1_summary.json")))
        got = json.loads(json.dumps(c1_summary({}, write=False)))
        if got != want:
            print("C1 summary differs", {k: (want.get(k), got.get(k)) for k in got if got.get(k) != want.get(k)})
            sys.exit(1)
        return
    os.makedirs(OUT, exist_ok=True)
    ledger = {"made_by": "tools/make_golden.py", "reference": "openjamoses/TOSEM-2021-Replication"}
    v1 = read_xlsx(os.path.join(REF, "Important-files/ML-Testing-v1.xlsx"), only=set(REV_A) | {"DeepSpeech"})
    golden_g4(v1, ledger)
    ledger_headers(v1, ledger)
    ledger_g1(v1, ledger)
    golden_g3(ledger)
    ledger_g2(ledger)
    c1_summary(ledger)
    ledger["C1"]["fixture"] = c1_fixture()
    ledger["C1"]["hazard_fixture"] = c1_hazards()
    json.dump(ledger, open(os.path.join(OUT, "ledger.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
