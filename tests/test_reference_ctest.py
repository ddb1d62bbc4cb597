"""The reference's OWN regression tests (its CMakeLists.txt and src/test/test.cmake: `diamond ARGS -o NAME.out` must equal the
expected NAME.out byte for byte) replayed through this repository's CLI over the oracle-linked host pipeline: every case whose
options the path implements.  These are the reference's known-answer vectors for the path (SURVEY 8c): real proteins (data.faa:
300 sequences; a sample of nr_10k.faa), its nanopore reads for blastx (FASTQ and gzipped FASTA), all sensitivity modes from the
default to --ultra-sensitive, -k / -e / --comp-based-stats 0, the pairwise format.  Inputs and command lines: tests/golden/refdata
(tests/golden/make_refdata.py); the reference's outputs on them: tests/golden/reference_outputs.json.  The live comparisons
further down run the reference's CLI on synthetic workloads, recorded the same way.  CPU only."""
import gzip, json, os, shutil, subprocess
import pytest
from conftest import GOLDEN, ROOT, reference_output, text_digest, workload_blocks

CLI = os.path.join(ROOT, "oracle", "_build", "dmnd-oracle-cli")
REFDATA = os.path.join(GOLDEN, "refdata")
COMMANDS = json.load(open(os.path.join(REFDATA, "ctest_commands.json")))  # {case: argument list with ${TD}}


@pytest.fixture(scope="session")
def td(tmp_path_factory):
    """The test inputs as the reference's command lines name them (FASTA, FASTQ and DAA files are stored gzip-compressed)."""
    d = tmp_path_factory.mktemp("refdata")
    for f in os.listdir(REFDATA):
        src = os.path.join(REFDATA, f)
        if f.endswith((".faa.gz", ".fastq.gz", ".daa.gz")):
            open(d / f[:-3], "wb").write(gzip.open(src).read())
        else:
            shutil.copy(src, d / f)
    return str(d)


@pytest.mark.parametrize("name", list(COMMANDS))
def test_reference_ctest_case(oracle_lib, td, name, tmp_path):
    args = [a.replace("${TD}", td) for a in COMMANDS[name]]
    if "nr_10k.dmnd" in args:  # (the reference's suite builds this database in an earlier test, with taxonomy files that do not enter the search; ours: plain makedb)
        db = str(tmp_path / "nr_10k")
        subprocess.run([CLI, "makedb", "--in", os.path.join(td, "nr_10k.faa"), "-d", db], capture_output=True, check=True)
        args = [db + ".dmnd" if a == "nr_10k.dmnd" else a for a in args]
    out = str(tmp_path / (name + ".out"))
    r = subprocess.run([CLI] + args + ["-o", out], capture_output=True, text=True)
    assert r.returncode == 0, " ".join(args) + "\n" + r.stderr
    want = reference_output("ctest/" + name, args)
    assert text_digest(open(out, "rb").read()) == want, " ".join(args)
    assert want["bytes"] > 0


@pytest.mark.parametrize("mode", ["blastp", "blastx"])
def test_paf_reports_unaligned_queries_like_the_reference(oracle_lib, mode, tmp_path):
    """PAF (Output::Flags::DEFAULT_REPORT_UNALIGNED): a query that had seed hits but no alignment gets the "4 *" record, a query
    without seed hits gets nothing (align/align.cpp:167-181, align/output.cpp:32-54) -- dmnd_result_unaligned.  A strict e-value
    makes many such queries; blastx adds the '-' strand and nucleotide coordinates."""
    from diamond_b200 import synth
    d = str(tmp_path / "d.faa")
    if mode == "blastp":
        w, *_ = workload_blocks("edge")
        q = str(tmp_path / "q.faa")
        synth.write_fasta(q, w["q_letters"], w["q_off"], "q")
        flags = ["--fast", "-e", "1e-40"]
    else:
        f, kw = synth.BX_WORKLOADS["bx"]
        w = f(**kw)
        q = str(tmp_path / "q.fna")
        synth.write_dna_fasta(q, w["dna"])
        flags = ["-e", "1e-30"]
    synth.write_fasta(d, w["db_letters"], w["db_off"], "d")
    ours = str(tmp_path / "o.paf")
    ref = reference_output(f"paf_unaligned/{mode}", [mode] + flags + ["-q", q, "-d", d, "-f", "paf", "-p", "8", "--quiet"])
    r = subprocess.run([CLI, mode] + flags + ["-q", q, "-d", d, "-f", "paf", "-o", ours, "-p", "8"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = open(ours).read()
    assert text_digest(got) == ref
    lines = got.splitlines()
    assert sum(l.split("\t")[1:3] == ["4", "*"] for l in lines) > 50 and sum(l.split("\t")[4] == "+" for l in lines) > 20
    if mode == "blastx":
        assert sum(l.split("\t")[4] == "-" for l in lines) > 20


@pytest.mark.parametrize("top,mode", [("50", ["--fast"])])
def test_top_percent_like_the_reference(oracle_lib, top, mode, tmp_path):
    """--top on protein families (hundreds of targets per query, several ranking chunks): score-ordered culling, the bit-score
    window, one pass of the outer loop (align/culling.cpp:90-141, align/extend.cpp:79-92,336); --top 100 = every target."""
    from diamond_b200 import synth
    w = synth.family_workload(n_fam=3, fam_size=250, n_q=40, seed=77, member_div=(0.02, 0.15), query_div=(0.03, 0.3))
    q, d, ours = (str(tmp_path / x) for x in ("q.faa", "d.faa", "o.tsv"))
    synth.write_fasta(q, w["q_letters"], w["q_off"], "q")
    synth.write_fasta(d, w["db_letters"], w["db_off"], "d")
    ref = reference_output(f"top/{top}", ["blastp"] + mode + ["-q", q, "-d", d, "--top", top, "-p", "8", "--quiet"])
    r = subprocess.run([CLI, "blastp"] + mode + ["-q", q, "-d", d, "--top", top, "-o", ours, "-p", "8"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert text_digest(open(ours).read()) == ref
    assert ref["lines"] > 5000


@pytest.mark.parametrize("mode", ["blastp", "blastx"])
def test_sam_format_like_the_reference(oracle_lib, mode, tmp_path):
    """-f sam (output/sam_format.cpp): CIGAR, the aligned query letters, NM / ZI / ZF / ZS and the MD string from the edit transcript,
    "4 *" records for queries with seed hits and no alignment.  Everything but the @PG header line (it quotes the program's own
    command line) must equal the reference's file."""
    from diamond_b200 import synth
    d = str(tmp_path / "d.faa")
    if mode == "blastp":
        w, *_ = workload_blocks("edge")
        q = str(tmp_path / "q.faa")
        synth.write_fasta(q, w["q_letters"], w["q_off"], "q")
    else:
        f, kw = synth.BX_WORKLOADS["bx"]
        w = f(**kw)
        q = str(tmp_path / "q.fna")
        synth.write_dna_fasta(q, w["dna"])
    synth.write_fasta(d, w["db_letters"], w["db_off"], "d")
    ours = str(tmp_path / "o.sam")
    flags = ["--fast", "-e", "1e-15", "-q", q, "-d", d, "-f", "sam", "-p", "8"]
    ref = reference_output(f"sam/{mode}", [mode] + flags + ["--quiet"], drop_prefix="@PG")
    r = subprocess.run([CLI, mode] + flags + ["-o", ours], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    a = [l for l in open(ours) if not l.startswith("@PG")]
    assert text_digest("".join(a)) == ref and len(a) > 100
    assert any("^" in l.split("MD:Z:")[1] for l in a if "MD:Z:" in l) or mode == "blastp"
    assert sum(l.split("\t")[1:3] == ["4", "*"] for l in a) > 10


@pytest.mark.parametrize("mode", ["blastp", "blastx"])
def test_more_tabular_fields_like_the_reference(oracle_lib, td, mode, tmp_path):
    """qtitle / stitle (first title of a merged record), positive / ppos, qcovhsp / scovhsp, qframe / qstrand, qseq (the read's nucleotides for blastx) / sseq, with --unal 1, on the
    reference's real test data (samples of the nr_300 proteins / nanopore reads against nr_10k)."""
    fields = "qseqid qtitle sseqid stitle pident positive ppos qcovhsp scovhsp qframe qstrand length evalue qseq sseq".split()
    if mode == "blastp":
        q = os.path.join(td, "nr_300.faa")
    else:
        q = str(tmp_path / "nano.fna")
        open(q, "wb").write(gzip.open(os.path.join(td, "SRR14011045_1.fna.gz")).read())
    flags = ["--fast", "-q", q, "-d", os.path.join(td, "nr_10k.faa"), "-p", "8", "--unal", "1", "--header", "simple", "-e", "1e-10", "-f", "6"] + fields
    ours = str(tmp_path / "o.tsv")
    ref = reference_output(f"more_tabular_fields/{mode}", [mode] + flags + ["--quiet"])
    r = subprocess.run([CLI, mode] + flags + ["-o", ours], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = open(ours).read()
    assert text_digest(got) == ref and got.count("\n") > 20


@pytest.mark.parametrize("extra", [["-c1", "-b0.00002"], ["--fast", "-b0.00003", "--top", "10"], ["-b0.00005", "-k", "3", "-f", "6", "qseqid", "sseqid", "evalue", "bitscore", "cigar"]])
def test_blocked_dmnd_database_matches_reference(oracle_lib, td, extra, tmp_path):
    """Reference blocks of a .dmnd database are cut by LETTERS (SequenceFile::load_twopass), FASTA databases by file bytes (the two
    ctest cases above): our -b on a DIAMOND database file against the reference binary, incl. --top (join by score) and transcripts
    carried through the join.  The database is written by our makedb, which the reference read for the recording; that our makedb
    writes the reference's file byte for byte is test_masking.py::test_makedb_and_dmnd_reader."""
    db = str(tmp_path / "db")
    subprocess.run([CLI, "makedb", "--in", os.path.join(td, "data.faa"), "-d", db], check=True, capture_output=True)
    ref = reference_output("blocked_dmnd/" + " ".join(extra), ["blastp", "-q", os.path.join(td, "data.faa"), "-d", db, "-p4"] + extra + ["--quiet"])
    out = str(tmp_path / "o.out")
    r = subprocess.run([CLI, "blastp", "-q", os.path.join(td, "data.faa"), "-d", db + ".dmnd", "-p4", "-o", out] + extra, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert text_digest(open(out, "rb").read()) == ref and ref["bytes"] > 1000
