#!/usr/bin/env python3
"""Write the stored results that three tests compare with when the reference's own programs are not built into
oracle/_ref/ (which needs the reference sources, see oracle/Makefile):

  tests/golden/ref_cpu_scan_live.json   scores of tests/test_oracle.py::test_oracle_scan_matches_reference_cpu_routine_live
  tests/golden/align/<matrix>.tsv       `align` results of tests/test_cli.py::test_align_matches_reference_align
  tests/golden/align/pseudodb.txt       `align` results of tests/test_cli.py::test_align_plain_output_and_pseudodb

They are outputs of this project's own code (the CPU oracle and `build/align`), which these tests compared byte for
byte with the reference's CPU routine and `align` binary while those were built. Every top-k list written here is
checked against the CPU oracle first.

  python tools/make_golden_outputs.py [cpu] [align]      (default: both; `align` needs a GPU and a built tree)
"""
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cudasw4_b200 import dbformat  # noqa: E402
from tests import oracle_lib, test_cli, test_oracle  # noqa: E402

G = os.path.join(ROOT, "tests", "golden")
DEFAULT_GAPS = {45: (-13, -2), 50: (-13, -2), 62: (-11, -1), 80: (-10, -1)}  # align's per-matrix defaults


def cpu(oracle):
    db, cases = test_oracle.live_scan_cases()
    out = [{"query_length": len(q), "gop": gop, "gex": gex, "scores": oracle.scan(62, q, db, gop, gex).tolist()}
           for q, gop, gex in cases]
    with open(os.path.join(G, "ref_cpu_scan_live.json"), "w") as f:
        json.dump({"source": "oracle/sw_oracle.cpp (BLOSUM62); the test compared it on these inputs with the reference's "
                             "scalar CPU Gotoh (src/cudasw4.cuh:2331-2392) while that was built", "cases": out}, f)


def _run(args, cwd):
    subprocess.run([test_cli.ALIGN] + args, cwd=cwd, check=True, stdout=subprocess.DEVNULL)
    return open(os.path.join(cwd, args[args.index("--of") + 1])).read()


def align(oracle):
    os.makedirs(os.path.join(G, "align"), exist_ok=True)
    for mat, extra in test_cli.ALIGN_CASES:
        with tempfile.TemporaryDirectory() as tmp:
            common = test_cli.align_case_inputs(tmp, mat, extra)
            tsv = _run(common + ["--dpx", "--of", "ours.tsv"], tmp)
            blosum = int(mat[len("blosum"):])
            gop, gex = DEFAULT_GAPS[blosum]
            if extra:
                gop, gex = int(extra[extra.index("--gop") + 1]), int(extra[extra.index("--gex") + 1])
            db = dbformat.read_db(os.path.join(tmp, "db"))
            rows = [r.split("\t") for r in tsv.splitlines()[1:]]
            for qi, (_, q) in enumerate(dbformat.read_fasta(os.path.join(tmp, "q.fa"))):
                s, i = oracle.topk(oracle.scan(blosum, dbformat.encode(q), db, gop, gex), 25)
                mine = [r for r in rows if int(r[0]) == qi]
                assert [int(r[4]) for r in mine] == s.tolist() and [int(r[7]) for r in mine] == i.tolist(), (mat, qi)
        with open(os.path.join(G, "align", f"{mat}.tsv"), "w") as f:
            f.write(tsv)
    with tempfile.TemporaryDirectory() as tmp:
        txt = _run(test_cli.pseudodb_case_inputs(tmp) + ["--of", "res.txt"], tmp)
    # every PseudoDB subject is the same sequence, so each query's top 3 are ids 0..2 with its known score (SURVEY.md 8c)
    with open(os.path.join(G, "survey_kat.json")) as f:
        kat = json.load(f)["pseudodb_blosum62_gop-11_gex-1"]["256"]
    lines = txt.splitlines()
    assert len(lines) == 8
    for qi in range(2):
        assert all(f"Score: {kat[qi]}. Length: 256. Header H. referenceId {r}" in lines[4 * qi + 1 + r] for r in range(3))
    with open(os.path.join(G, "align", "pseudodb.txt"), "w") as f:
        f.write(txt)


def main():
    parts = sys.argv[1:] or ["cpu", "align"]
    oracle = oracle_lib.load()
    for p in parts:
        {"cpu": cpu, "align": align}[p](oracle)
    print("written under", G)


if __name__ == "__main__":
    main()
