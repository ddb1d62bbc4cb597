"""Masking parity (SURVEY 8f rank 2 -> the reference's DEFAULT flags): tantan hard masking of both blocks
(masking/tantan.cpp) and motif soft masking (masking/masking.cpp:110-131) in the oracle, pinned against the reference:
 * fmt-6 + --log counters of the L2 goldens (tests/golden/*.l2.*: the reference run with its default flags);
 * the tantan lambda constant against the value the reference's own LambdaCalculator.cc derives (tests/golden/tantan_lambda.txt;
   compiled from the reference's sources and derived again where DMND_REFERENCE_SRC names a checkout of it);
 * the reference's default-flag output on real proteins (a sample of its src/test/nr_10k.faa, X/B/J letters), as recorded in
   tests/golden/reference_outputs.json.
CPU only."""
import ctypes as C, json, os, re, subprocess, tempfile
import numpy as np
import pytest
from conftest import GOLDEN, ROOT, reference_output, text_digest, workload_blocks

WORKLOADS = ["c1", "fam2", "edge", "long", "rep"]


@pytest.mark.parametrize("name", WORKLOADS)
def test_default_flags_match_reference_golden(oracle_lib, name):
    from diamond_b200 import api
    w, q_raw, q_lim, r_raw, r_lim = workload_blocks(name)
    ctx = api.Context(oracle_lib, threads=8, comp_based_stats=1, masking=1, motif_masking=1)
    m, _, st = ctx.blastp(q_raw, q_lim, r_raw, r_lim)
    ctx.close()
    assert api.fmt6(m) == open(os.path.join(GOLDEN, f"{name}.l2.tsv")).read()
    cn = json.load(open(os.path.join(GOLDEN, f"{name}.l2.counters.json")))
    for k in ("seeds_hit", "seed_hits", "tentative_matches1", "tentative_matches2", "tentative_matches3"):
        assert st["seed"][k] == cn[k], k
    assert st["targets"] == cn["targets"] and st["dp_problems_round2"] == cn["targets_round2"]


def test_repeat_workload_is_actually_masked(oracle_lib):
    """The fixture must exercise the code: tantan masks thousands of letters, the motif table marks ranges, and both change the output."""
    from diamond_b200 import api
    w, q_raw, q_lim, r_raw, r_lim = workload_blocks("rep")
    ctx = api.Context(oracle_lib, threads=8)
    rb = ctx.upload(r_raw, r_lim)
    pos = ctx.mask_block(rb, 5, 0, len(r_lim) - 1)
    after = ctx.download_letters(rb, r_raw.size)
    ctx.free_block(rb); ctx.close()
    assert len(pos) > 2000 and np.all(np.diff(pos.astype(np.int64)) > 0)
    changed = np.flatnonzero(after != r_raw)
    p64 = pos.astype(np.int64)
    assert np.all(after[p64] == 23) and np.all(np.isin(changed, p64))   # (a letter that already was X may be reported as well)
    assert np.all(r_raw[np.setdiff1d(p64, changed)] == 23)
    assert open(os.path.join(GOLDEN, "rep.l2.tsv")).read() != open(os.path.join(GOLDEN, "rep.l1.tsv")).read()


def test_resident_blocks_masked_by_the_caller_equal_the_e2e_call(oracle_lib):
    """dmnd_blastp masks inside the call; dmnd_blastp_resident expects masked blocks + equally masked host letters."""
    from diamond_b200 import api
    w, q_raw, q_lim, r_raw, r_lim = workload_blocks("rep")
    ctx = api.Context(oracle_lib, threads=8, comp_based_stats=1, masking=1, motif_masking=1)
    qb, rb = ctx.upload(q_raw, q_lim), ctx.upload(r_raw, r_lim)
    ctx.mask_block(qb, 5, 0, len(q_lim) - 1); ctx.mask_block(rb, 5, 0, len(r_lim) - 1)
    qm, rm = ctx.download_letters(qb, q_raw.size), ctx.download_letters(rb, r_raw.size)
    m, _, _ = ctx.blastp_resident(qb, rb, qm, q_lim, rm, r_lim)
    out = api.fmt6(m)
    ctx.free_block(qb); ctx.free_block(rb); ctx.close()
    assert out == open(os.path.join(GOLDEN, "rep.l2.tsv")).read()


@pytest.mark.parametrize("lanes", ["3"])
def test_query_lanes_mask_their_own_ranges(oracle_lib, lanes, monkeypatch):
    from diamond_b200 import api
    monkeypatch.setenv("DMND_LANES", lanes)
    w, q_raw, q_lim, r_raw, r_lim = workload_blocks("rep")
    ctx = api.Context(oracle_lib, threads=8, comp_based_stats=1, masking=1, motif_masking=1)
    m, _, _ = ctx.blastp(q_raw, q_lim, r_raw, r_lim)
    ctx.close()
    assert api.fmt6(m) == open(os.path.join(GOLDEN, "rep.l2.tsv")).read()


def test_tantan_lambda_equals_the_reference_lambda_calculator(oracle_lib, tmp_path):
    """dmnd_params_init hard-codes lambda(BLOSUM62 20x20) = 0x1.4bcf16a672882p-2: the value the reference's own
    lib/tantan/LambdaCalculator.cc derives (tests/golden/tantan_lambda.txt; re-derived from the reference's sources where
    DMND_REFERENCE_SRC names a checkout of it); the likelihood-ratio table is compared bit for bit."""
    from diamond_b200 import api
    o = api.SearchOpts(); oracle_lib.dmnd_search_opts_default(C.byref(o))
    p = api.Params(); assert oracle_lib.dmnd_params_init(C.byref(o), C.byref(p)) == 0
    s = list(p.score)
    lam = float.fromhex(open(os.path.join(GOLDEN, "tantan_lambda.txt")).read().split()[0])
    if os.environ.get("DMND_REFERENCE_SRC"):
        lam = _reference_lambda(os.path.join(os.environ["DMND_REFERENCE_SRC"], "src", "lib", "tantan"), s, tmp_path)
    assert lam == float.fromhex("0x1.4bcf16a672882p-2")
    lr = np.array(list(p.tantan_lr), dtype=np.float32).reshape(32, 32)
    want = np.zeros((32, 32), dtype=np.float32)
    for a in range(26):
        for b in range(26):
            want[a, b] = np.float32(np.exp(lam * s[a * 32 + b]))
    assert np.array_equal(lr.view(np.uint32), want.view(np.uint32))
    assert o.masking == 1 and o.motif_masking == 1  # the C defaults are the reference's defaults


def _reference_lambda(tantan, s, tmp_path):
    """lambda of the 20x20 part of the score matrix s by the reference's LambdaCalculator, compiled from its sources."""
    src = tmp_path / "probe.cpp"
    src.write_text('#include "LambdaCalculator.hh"\n#include <cstdio>\nint main(){int m[20][20];const int*p[20];for(int i=0;i<20;++i){p[i]=m[i];'
                   'for(int j=0;j<20;++j)if(scanf("%d",&m[i][j])!=1)return 2;}cbrc::LambdaCalculator lc;lc.calculate(p,20);printf("%a\\n",lc.lambda());return 0;}\n')
    exe = tmp_path / "probe"
    subprocess.run(["g++", "-O2", "-I" + tantan, str(src), os.path.join(tantan, "LambdaCalculator.cc"), "-o", str(exe)], check=True)
    txt = "\n".join(" ".join(str(s[a * 32 + b]) for b in range(20)) for a in range(20))
    return float.fromhex(subprocess.run([str(exe)], input=txt, capture_output=True, text=True, check=True).stdout.strip())


NR10K = os.path.join(GOLDEN, "refdata", "nr_10k.faa.gz")  # a sample of the reference's nr_10k.faa


def test_live_reference_default_flags_on_real_proteins(tmp_path):
    """Real proteins (X, B, J letters, long viral polyproteins that are > 50 % motif-covered) against themselves with
    the reference's default flags: fmt-6 byte-identical and the --log stage counters equal."""
    import gzip
    cli = os.path.join(ROOT, "oracle", "_build", "dmnd-oracle-cli")
    sub = tmp_path / "nr.faa"
    sub.write_bytes(gzip.open(NR10K).read())
    our_out = tmp_path / "our.tsv"
    pats = (r"Seeds hit\s+= (\d+)", r"Hits \(filter stage 0\) = (\d+)", r"Hits \(filter stage 1\) = (\d+)", r"Hits \(filter stage 3\) = (\d+)", r"Target hits \(stage 0\) = (\d+)")
    ref = reference_output("real_proteins/fast", ["blastp", "--fast", "-q", str(sub), "-d", str(sub), "-f", "6", "-p", "8", "--log"], pats)
    o = subprocess.run([cli, "blastp", "--fast", "-q", str(sub), "-d", str(sub), "-o", str(our_out), "-p", "8", "--log"], capture_output=True, text=True, check=True)
    assert text_digest(our_out.read_text(), o.stdout + o.stderr, pats) == ref and ref["bytes"] > 10000


def _fasta_blocks(path, limit):
    import gzip
    from diamond_b200 import api
    alph = {c: i for i, c in enumerate("ARNDCQEGHILKMFPSTWYVBJZX*_")}
    seqs, cur = [], []
    for line in gzip.open(path, "rt"):
        if line.startswith(">"):
            if cur:
                seqs.append("".join(cur)); cur = []
            if len(seqs) >= limit:
                break
        else:
            cur.append(line.strip())
    if cur and len(seqs) < limit:
        seqs.append("".join(cur))
    letters = np.array([alph.get(c.upper(), 23) for s in seqs for c in s], dtype=np.int8)
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    np.cumsum([len(s) for s in seqs], out=off[1:])
    return api.block_image(letters, off)


@pytest.mark.parametrize("source", ["synthetic", "rep", "nr10k"])
def test_forward_only_certificate_is_sound(oracle_lib, source):
    """The device skips tantan's backward pass for sequences whose total HMM weight Z stays below 8x the all-background
    weight (log2 ratio < 3, mask_kernels.cuh): then no letter can reach the 0.9 masking threshold.  Checked against the full
    computation of the oracle: every sequence below the bound has no masked letter; and the bound is worth having."""
    from diamond_b200 import api, synth
    if source == "nr10k":
        raw, lim = _fasta_blocks(NR10K, 4000)
    elif source == "rep":
        raw, lim = workload_blocks("rep")[3:5]
    else:
        w = synth.workload(100, 20000, 7)
        raw, lim = api.block_image(w["db_letters"], w["db_off"])
    n = len(lim) - 1
    ctx = api.Context(oracle_lib, threads=8)
    b = ctx.upload(raw, lim)
    ratio, masked = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.uint32)
    oracle_lib.dmnd_oracle_tantan_log2_ratio.argtypes = [C.c_void_p] * 4
    assert oracle_lib.dmnd_oracle_tantan_log2_ratio(ctx.ctx, b, ratio.ctypes.data, masked.ctypes.data) == 0
    ctx.free_block(b); ctx.close()
    lens = np.diff(lim) - 1
    cert = (ratio < 3.0) & (lens <= 4096)
    assert not np.any(masked[cert] > 0), f"{int((masked[cert] > 0).sum())} certified sequences have masked letters"
    assert np.all(ratio[lens > 0] > -1e-3)  # Z >= W_bg
    if source == "synthetic":
        assert cert.mean() > 0.85
    print(source, "certified", float(cert.mean()), "masked seqs", int((masked > 0).sum()), "closest call", float(ratio[masked > 0].min()) if (masked > 0).any() else None)


@pytest.mark.parametrize("name", ["c1", "edge", "long", "rep"])
def test_transcript_fields_match_reference_golden(oracle_lib, name, tmp_path):
    """north_star: CIGAR / traceback bit-exact.  The CLI's cigar, btop, qseq_gapped and sseq_gapped columns (built from the
    library's edit transcripts and its list of masked letters) against the reference's own columns (T2 goldens; `long` =
    7-12 k-letter proteins traced back, `rep` = masked letters inside alignments)."""
    from diamond_b200 import synth
    w, *_ = workload_blocks(name)
    q, d, o = (str(tmp_path / x) for x in ("q.faa", "d.faa", "o.tsv"))
    synth.write_fasta(q, w["q_letters"], w["q_off"], "q")
    synth.write_fasta(d, w["db_letters"], w["db_off"], "d")
    cli = os.path.join(ROOT, "oracle", "_build", "dmnd-oracle-cli")
    fields = "qseqid sseqid pident length mismatch gapopen qstart qend sstart send evalue bitscore cigar btop qseq_gapped sseq_gapped".split()
    r = subprocess.run([cli, "blastp", "--fast", "-q", q, "-d", d, "-f", "6"] + fields + ["-o", o, "-p", "8"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    gold = open(os.path.join(GOLDEN, f"{name}.t2.tsv")).read()
    assert open(o).read() == gold
    if name != "long":  # (with a transcript the reference traces the > 10^6-cell problems of `long` back instead of running its statistics passes: one mismatch count differs)
        assert [l.split("\t")[:12] for l in gold.splitlines()] == [l.split("\t") for l in open(os.path.join(GOLDEN, f"{name}.l2.tsv")).read().splitlines()]
    if name == "rep":
        assert any("X" in l.split("\t")[13] for l in gold.splitlines())  # masked letters do show up in BTOP


@pytest.mark.parametrize("name", ["edge", "long"])
def test_pairwise_format_matches_reference_golden(oracle_lib, name, tmp_path):
    """-f 0, the BLAST pairwise format (output/blast_pairwise_format.cpp:24-101): header, query intros, 60-column alignment
    blocks with midline, identities / positives / gaps -- from the library's transcripts; byte-identical to the reference's file."""
    from diamond_b200 import synth
    w, *_ = workload_blocks(name)
    q, d, o = (str(tmp_path / x) for x in ("q.faa", "d.faa", "o.txt"))
    synth.write_fasta(q, w["q_letters"], w["q_off"], "q")
    synth.write_fasta(d, w["db_letters"], w["db_off"], "d")
    cli = os.path.join(ROOT, "oracle", "_build", "dmnd-oracle-cli")
    r = subprocess.run([cli, "blastp", "--fast", "-q", q, "-d", d, "-f", "0", "-o", o, "-p", "8"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(o).read() == open(os.path.join(GOLDEN, f"{name}.f0.txt")).read()


def test_makedb_and_dmnd_reader(oracle_lib, tmp_path):
    """`makedb` writes the reference's database format byte for byte (legacy/dmnd: headers, MurmurHash3 database hash, records
    with the tantan soft-mask bit from dmnd_block_mask, position array) -- tests/golden/rep100.dmnd is the reference's own
    makedb output for the first 100 sequences of the `rep` database -- and `blastp -d` reads such a file back: same output as
    with the FASTA database."""
    from diamond_b200 import synth
    w, *_ = workload_blocks("rep")
    d100, q = str(tmp_path / "d100.faa"), str(tmp_path / "q.faa")
    synth.write_fasta(d100, w["db_letters"][: w["db_off"][100]], w["db_off"][:101], "d")
    synth.write_fasta(q, w["q_letters"], w["q_off"], "q")
    cli = os.path.join(ROOT, "oracle", "_build", "dmnd-oracle-cli")
    r = subprocess.run([cli, "makedb", "--in", d100, "-d", str(tmp_path / "ours")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    ours, gold = open(tmp_path / "ours.dmnd", "rb").read(), open(os.path.join(GOLDEN, "rep100.dmnd"), "rb").read()
    assert ours == gold and sum(1 for b in gold[96:] if b & 0x80 and b != 0xff) > 100  # (soft-mask bits are present)
    out = []
    for db in (d100, str(tmp_path / "ours.dmnd"), str(tmp_path / "ours")):  # FASTA, .dmnd, .dmnd without the extension
        o = str(tmp_path / "o.tsv")
        r = subprocess.run([cli, "blastp", "--fast", "-q", q, "-d", db, "-o", o, "-p", "8"], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        out.append(open(o).read())
    assert out[0] == out[1] == out[2] and out[0].count("\n") > 10
    r = subprocess.run([cli, "makedb", "--in", d100, "-d", str(tmp_path / "x"), "--masking", "0"], capture_output=True, text=True)
    assert r.returncode != 0 and "not permitted" in r.stderr


def test_reference_reads_our_database(oracle_lib, tmp_path):
    """The unmodified reference searches a database written by our makedb and gives the L2 golden (its output is stored under
    the digest of the database file it read: a makedb that writes another file has no stored output)."""
    import hashlib
    from diamond_b200 import synth
    w, *_ = workload_blocks("edge")
    d, q, o = (str(tmp_path / x) for x in ("d.faa", "q.faa", "o.tsv"))
    synth.write_fasta(d, w["db_letters"], w["db_off"], "d")
    synth.write_fasta(q, w["q_letters"], w["q_off"], "q")
    cli = os.path.join(ROOT, "oracle", "_build", "dmnd-oracle-cli")
    subprocess.run([cli, "makedb", "--in", d, "-d", str(tmp_path / "db")], capture_output=True, check=True)
    db = hashlib.sha256(open(tmp_path / "db.dmnd", "rb").read()).hexdigest()
    ref = reference_output("reads_our_database/" + db, ["blastp", "--fast", "-q", q, "-d", str(tmp_path / "db.dmnd"), "-f", "6", "-p", "8", "--quiet"])
    assert ref == text_digest(open(os.path.join(GOLDEN, "edge.l2.tsv")).read())
