"""Drop-in CLIs. CPU: our makedb reproduces the reference makedb's files byte for byte (golden fixtures written by the
reference binary). GPU: our `align` prints the same result files as the reference's own `align` (--dpx and default
half2 kernels) on the same database and queries: the stored results under tests/golden/align/, and live when the
reference has been built into oracle/_ref/ (oracle/Makefile)."""
import os
import subprocess

import numpy as np
import pytest

from cudasw4_b200 import dbformat, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAKEDB = os.path.join(ROOT, "build", "makedb")
ALIGN = os.path.join(ROOT, "build", "align")
REF_ALIGN = os.path.join(ROOT, "oracle", "_ref", "align_gapfix")


def _build_cli():
    if not (os.path.exists(MAKEDB) and os.path.exists(ALIGN)):
        env = {k: v for k, v in os.environ.items() if k not in ("CXX", "CC")}
        subprocess.run(["make", "-C", ROOT, "cli"], check=True, env=env, stdout=subprocess.DEVNULL)


def test_makedb_matches_reference_makedb(golden_dir, tmp_path):
    _build_cli()
    for name in ("tinydb", "tiesdb"):
        out = str(tmp_path / name)
        os.makedirs(out)
        subprocess.run([MAKEDB, os.path.join(golden_dir, name, "input.fasta"), os.path.join(out, "db")], check=True,
                       stdout=subprocess.DEVNULL)
        for suffix in ("0chars", "0offsets", "0lengths", "0headers", "0headeroffsets", "0metadata", "metadata"):
            with open(os.path.join(golden_dir, name, "db" + suffix), "rb") as a, open(os.path.join(out, "db" + suffix), "rb") as b:
                assert a.read() == b.read(), (name, suffix)


def test_makedb_gzip_and_fastq(tmp_path):
    _build_cli()
    import gzip
    recs = [("r1 desc", "ARNDCQEGHILKMFPSTWYV"), ("r2", "WWXBZ"), ("r3", "AC")]
    fq = tmp_path / "in.fastq.gz"
    with gzip.open(fq, "wt") as f:
        for h, s in recs:
            f.write(f"@{h}\n{s}\n+\n{'I' * len(s)}\n")
    subprocess.run([MAKEDB, str(fq), str(tmp_path / "db")], check=True, stdout=subprocess.DEVNULL)
    db = dbformat.read_db(str(tmp_path / "db"))
    assert db.lengths.tolist() == [2, 5, 20]
    assert [db.header(i) for i in range(3)] == ["r3", "r2", "r1 desc"]
    assert dbformat.decode(db.sequence(1)) == "WW---"


def _run_align(binary, args, cwd):
    r = subprocess.run([binary] + args, cwd=cwd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:] + r.stdout[-2000:]
    return r.stdout


ALIGN_CASES = [("blosum62", []), ("blosum45", []), ("blosum80", ["--gop", "-14", "--gex", "-2"])]


def align_case_inputs(workdir, mat, extra):
    """Writes the database and queries of test_align_matches_reference_align into `workdir` (with the makedb files of
    the database under the prefix `db`); returns the `align` arguments the test runs both programs with."""
    _build_cli()
    recs, queries = synth.config_c1(seed=1, n=3000)
    rng = np.random.default_rng(5)
    recs += [(f"long{i}", dbformat.decode(synth.random_residues(rng, int(n)))) for i, n in enumerate([1300, 2000, 4100, 8100, 9000])]
    dbformat.write_fasta(os.path.join(workdir, "db.fa"), recs)
    dbformat.write_fasta(os.path.join(workdir, "q.fa"), queries[:6] + [queries[19]])
    subprocess.run([MAKEDB, os.path.join(workdir, "db.fa"), os.path.join(workdir, "db")], check=True, stdout=subprocess.DEVNULL)
    return ["--query", "q.fa", "--db", "db", "--top", "25", "--tsv", "--mat", mat, "--uploadFull", "--prefetchDBFile"] + extra


def pseudodb_case_inputs(workdir):
    """Writes the queries of test_align_plain_output_and_pseudodb into `workdir`; returns the common `align` arguments."""
    _build_cli()
    dbformat.write_fasta(os.path.join(workdir, "q.fa"), synth.load_queries()[:2])
    return ["--query", "q.fa", "--pseudodb", "5000", "256", "--top", "3"]


@pytest.mark.gpu
@pytest.mark.parametrize("mat,extra", ALIGN_CASES)
def test_align_matches_reference_align(tmp_path, golden_dir, mat, extra):
    common = align_case_inputs(str(tmp_path), mat, extra)
    _run_align(ALIGN, common + ["--dpx", "--of", "ours.tsv"], str(tmp_path))
    ours = open(tmp_path / "ours.tsv").read()
    assert ours.count("\n") == 1 + 7 * 25
    with open(os.path.join(golden_dir, "align", f"{mat}.tsv")) as f:
        assert ours == f.read()
    if not os.path.exists(REF_ALIGN):
        return
    for tag, flags in (("dpx", ["--dpx"]), ("half2", [])):
        _run_align(REF_ALIGN, common + flags + ["--of", f"ref_{tag}.tsv"], str(tmp_path))
        ref = open(tmp_path / f"ref_{tag}.tsv").read()
        assert ours == ref, tag


@pytest.mark.gpu
def test_align_plain_output_and_pseudodb(tmp_path, golden_dir):
    common = pseudodb_case_inputs(str(tmp_path))
    out = _run_align(ALIGN, common + ["--verbose", "--of", "res.txt"], str(tmp_path))
    assert "Total time:" in out and "GCUPS" in out
    res = open(tmp_path / "res.txt").read().splitlines()
    assert res[0].startswith("Query 0, header") and ", num overflows 0" in res[0]
    assert res[1] == "Result 0. Score: 25. Length: 256. Header H. referenceId 0"
    assert res[3] == "Result 2. Score: 25. Length: 256. Header H. referenceId 2"
    with open(os.path.join(golden_dir, "align", "pseudodb.txt")) as f:
        assert open(tmp_path / "res.txt").read() == f.read()
    if os.path.exists(REF_ALIGN):
        _run_align(REF_ALIGN, common + ["--dpx", "--uploadFull", "--of", "ref.txt"], str(tmp_path))
        assert open(tmp_path / "ref.txt").read() == open(tmp_path / "res.txt").read()


@pytest.mark.gpu
def test_align_batch_queries_and_streaming_write_the_same_file(tmp_path):
    """--batchQueries (several scans in flight, sw4_scan_many) and --maxGpuMem small enough to stream the database in
    batches must produce byte-identical result files to the plain one-query-at-a-time resident run."""
    _build_cli()
    recs, queries = synth.config_c1(seed=2, n=12000)
    dbformat.write_fasta(str(tmp_path / "db.fa"), recs)
    dbformat.write_fasta(str(tmp_path / "q.fa"), queries[:9])
    subprocess.run([MAKEDB, str(tmp_path / "db.fa"), str(tmp_path / "db")], check=True, stdout=subprocess.DEVNULL)
    common = ["--query", "q.fa", "--db", "db", "--top", "12", "--mat", "blosum62", "--dpx"]
    _run_align(ALIGN, common + ["--of", "plain.txt"], str(tmp_path))
    _run_align(ALIGN, common + ["--of", "batched.txt", "--batchQueries", "4"], str(tmp_path))
    _run_align(ALIGN, common + ["--of", "streamed.txt", "--maxGpuMem", "5M", "--batchQueries", "16", "--verbose"], str(tmp_path))
    plain = open(tmp_path / "plain.txt").read()
    assert plain.count("Query ") == 9
    assert open(tmp_path / "batched.txt").read() == plain
    assert open(tmp_path / "streamed.txt").read() == plain
