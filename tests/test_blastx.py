"""blastx (SURVEY 8f rank 3): DNA queries translated into six frames per read, searched with the unchanged K layer, extended
per frame with the reference's frame-aware target logic (align/ungapped.cpp:76-116, gapped_score.cpp:107-246, culling.cpp:58-67)
and reported in nucleotide coordinates.  Goldens: tests/golden/bx.x0 / bx.xt = the unmodified reference, `blastx --fast`,
default flags (tantan + motif masking of the translated frames, Hauser CBS), on synth.BX_WORKLOADS.  CPU only: the host
pipeline over the oracle's K layer."""
import json, os, subprocess
import numpy as np
import pytest
from conftest import GOLDEN, ROOT, reference_output, text_digest

CLI = os.path.join(ROOT, "oracle", "_build", "dmnd-oracle-cli")
XT_FIELDS = "qseqid sseqid pident length mismatch gapopen qstart qend sstart send evalue bitscore cigar btop qseq_gapped sseq_gapped score qlen slen".split()


def _bx():
    from diamond_b200 import synth
    f, kw = synth.BX_WORKLOADS["bx"]
    return f(**kw)


def _files(w, tmp_path):
    from diamond_b200 import synth
    q, d = str(tmp_path / "q.fna"), str(tmp_path / "d.faa")
    synth.write_dna_fasta(q, w["dna"])
    synth.write_fasta(d, w["db_letters"], w["db_off"], "d")
    return q, d


@pytest.mark.parametrize("lanes", ["1", "3"])
def test_blastx_library_matches_reference_golden(oracle_lib, lanes, monkeypatch):
    """Through the C ABI: query block = api.translate_reads (six contexts per read), opts.query_contexts = 6."""
    from diamond_b200 import api
    monkeypatch.setenv("DMND_LANES", lanes)
    w = _bx()
    ql, qo = api.translate_reads(w["dna"])
    assert len(qo) - 1 == 6 * len(w["dna"])
    q_raw, q_lim = api.block_image(ql, qo)
    r_raw, r_lim = api.block_image(w["db_letters"], w["db_off"])
    g = api.Context(lib=oracle_lib, masking=1, motif_masking=1, query_contexts=6)
    m, _, st = g.blastp(q_raw, q_lim, r_raw, r_lim)
    g.close()
    assert api.fmt6_translated(m, [len(r) for r in w["dna"]]) == open(os.path.join(GOLDEN, "bx.x0.tsv")).read()
    gold = json.load(open(os.path.join(GOLDEN, "bx.x0.counters.json")))
    keys = ("seeds_hit", "seed_hits", "tentative_matches3") if lanes == "1" else ("seed_hits", "tentative_matches3")  # (a seed shared by two lanes counts in both)
    assert {k: st["seed"][k] for k in keys} == {k: gold[k] for k in keys}
    assert st["targets"] == gold["targets"] and st["targets_extended"] == gold["targets_extended"]
    frames = np.bincount(m["query"] % 6, minlength=6)
    assert frames.min() > 0  # every frame of either strand produced alignments
    per_read = {}
    for x in m:
        per_read.setdefault(int(x["query"]) // 6, set()).add(int(x["query"]) % 6)
    assert any(len(v) > 1 for v in per_read.values())  # chimeric / frame-shifted reads: one read reports targets in several frames


def test_blastx_cli_default_fields(oracle_lib, tmp_path):
    q, d = _files(_bx(), tmp_path)
    o = str(tmp_path / "o.tsv")
    r = subprocess.run([CLI, "blastx", "--fast", "-q", q, "-d", d, "-o", o, "-p", "8"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(o).read() == open(os.path.join(GOLDEN, "bx.x0.tsv")).read()


def test_blastx_cli_transcript_fields(oracle_lib, tmp_path):
    """cigar / btop / gapped sequences of the translated frame (masked letters included), score, qlen in nucleotides."""
    q, d = _files(_bx(), tmp_path)
    o = str(tmp_path / "o.tsv")
    r = subprocess.run([CLI, "blastx", "--fast", "-q", q, "-d", d, "-f", "6"] + XT_FIELDS + ["-o", o, "-p", "8"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(o).read() == open(os.path.join(GOLDEN, "bx.xt.tsv")).read()


@pytest.mark.parametrize("lvl,flags", [("x1", []), ("x3", ["--sensitive"]), ("x5", ["--very-sensitive"])])
def test_blastx_modes_above_fast(oracle_lib, tmp_path, lvl, flags):
    """No flag = the default sensitivity, as most users run `diamond blastx`: translated frames of <= 85 letters take the
    stage-2 window over their whole length (search/stage2.h:58-63), --sensitive and above add the gapped filter with its
    exceptions for short translated queries (align/extend.cpp:197-206, gapped_filter.cpp:44-55), --very-sensitive reads
    cutoff_table_short for frames of 61..85 letters."""
    q, d = _files(_bx(), tmp_path)
    o = str(tmp_path / "o.tsv")
    r = subprocess.run([CLI, "blastx"] + flags + ["-q", q, "-d", d, "-o", o, "-p", "8", "--log"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(o).read() == open(os.path.join(GOLDEN, f"bx.{lvl}.tsv")).read()
    gold = json.load(open(os.path.join(GOLDEN, f"bx.{lvl}.counters.json")))
    import re
    got = {k: int(re.search(p, r.stderr).group(1)) for k, p in (("tentative_matches2", r"Hits \(filter stage 2\) = (\d+)"), ("tentative_matches3", r"Hits \(filter stage 3\) = (\d+)"),
                                                                  ("targets", r"Target hits \(stage 0\) = (\d+)"), ("targets_extended", r"Target hits \(stage 3\) = (\d+)"))}
    assert got == {k: gold[k] for k in got}
    if lvl != "x1":
        assert gold["targets_extended"] < gold["targets"]  # the gapped filter removed targets


def test_blastx_rejects_what_it_does_not_implement(oracle_lib, tmp_path):
    from diamond_b200 import api
    q, d = _files(_bx(), tmp_path)
    r = subprocess.run([CLI, "blastx", "--fast", "--range-culling", "-q", q, "-d", d, "-o", str(tmp_path / "o")], capture_output=True, text=True)
    assert r.returncode != 0 and "only supported in frameshift alignment mode" in r.stderr  # the reference's own rule (basic/config.cpp:824-825)
    r = subprocess.run([CLI, "blastx", "--fast", "--taxon-k", "1", "-q", q, "-d", d, "-o", str(tmp_path / "o")], capture_output=True, text=True)
    assert r.returncode != 0 and "unsupported option" in r.stderr
    r = subprocess.run([CLI, "blastx", "--fast", "--max-hsps", "3", "-q", q, "-d", d, "-o", str(tmp_path / "o")], capture_output=True, text=True)
    assert r.returncode != 0 and "only 1 is implemented" in r.stderr
    # the library: contexts other than 1 / 6, nq not a multiple, or a window-filter mode
    raw, lim = api.block_image(np.zeros(40, dtype=np.int8), np.array([0, 10, 20, 30, 40], dtype=np.int64))
    g = api.Context(lib=oracle_lib, query_contexts=6)
    with pytest.raises(api.DmndError):
        g.blastp(raw, lim, raw, lim)  # 4 sequences
    g.close()


def test_live_reference_nanopore_reads(oracle_lib, tmp_path):
    """The reference's own blastx test input (a sample of src/test/SRR14011045_1.fna.gz against a sample of nr_10k.faa,
    tests/golden/refdata): nanopore reads of 0.3-4 kb full of frame shifts, run here with --fast and the transcript fields."""
    import gzip
    q, d = str(tmp_path / "nano.fna"), str(tmp_path / "nr.faa")
    open(q, "wb").write(gzip.open(os.path.join(GOLDEN, "refdata", "SRR14011045_1.fna.gz")).read())
    open(d, "wb").write(gzip.open(os.path.join(GOLDEN, "refdata", "nr_10k.faa.gz")).read())
    ours = str(tmp_path / "o.tsv")
    ref = reference_output("nanopore_reads/fast_transcripts", ["blastx", "--fast", "-q", q, "-d", d, "-f", "6"] + XT_FIELDS + ["-p", "8", "--quiet"])
    r = subprocess.run([CLI, "blastx", "--fast", "-q", q, "-d", d, "-f", "6"] + XT_FIELDS + ["-o", ours, "-p", "8"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert text_digest(open(ours).read()) == ref and ref["lines"] > 20


@pytest.mark.parametrize("flags", [["--strand", "minus"], ["--strand", "plus", "--min-orf", "30"], ["--query-gencode", "4", "--min-orf", "1"],
                                   ["--unal", "1", "-e", "1e-30"], ["--top", "10"], ["-k", "0", "-c", "1"]])
def test_blastx_options_like_the_reference(oracle_lib, flags, tmp_path):
    """Translation options (frames of a strand that is not searched stay in the block as X, data/block/block.cpp:95-96; --min-orf
    overrides Config::min_orf_len; NCBI table 4 reads TGA as W), --unal 1 records in nucleotide terms, --top and -k 0: live
    against the reference's output on the `bx` reads."""
    q, d = _files(_bx(), tmp_path)
    ours = str(tmp_path / "o.tsv")
    fields = ["-f", "6", "qseqid", "sseqid", "pident", "length", "qstart", "qend", "sstart", "send", "evalue", "bitscore", "qlen", "btop"]
    ref = reference_output("blastx_options/" + " ".join(flags), ["blastx", "--fast", "-q", q, "-d", d, "-p", "8", "--quiet"] + flags + fields)
    r = subprocess.run([CLI, "blastx", "--fast", "-q", q, "-d", d, "-o", ours, "-p", "8"] + flags + fields, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = open(ours).read()
    assert text_digest(got) == ref and got.count("\n") > 300
    if "--unal" in flags:
        assert sum(l.split("\t")[1] == "*" for l in got.splitlines()) > 50
    if flags[:2] == ["--strand", "minus"]:
        assert all(int(l.split("\t")[4]) > int(l.split("\t")[5]) for l in got.splitlines())  # qstart > qend: reverse strand only


@pytest.mark.parametrize("mode", ["blastx", "blastp"])
def test_pairwise_format_translated_and_unaligned(oracle_lib, mode, tmp_path):
    """-f 0 for blastx (" Frame = n" / "-n", query numbering on the read, descending on the reverse strand) and the "No hits found"
    records of queries that had seed hits but no alignment (strict e-value), against the reference's file."""
    from diamond_b200 import synth
    from conftest import workload_blocks
    d = str(tmp_path / "d.faa")
    if mode == "blastx":
        w = _bx()
        q = str(tmp_path / "q.fna")
        synth.write_dna_fasta(q, w["dna"])
        flags = ["--fast", "-e", "1e-20"]
    else:
        w, *_ = workload_blocks("edge")
        q = str(tmp_path / "q.faa")
        synth.write_fasta(q, w["q_letters"], w["q_off"], "q")
        flags = ["--fast", "-e", "1e-40"]
    synth.write_fasta(d, w["db_letters"], w["db_off"], "d")
    ours = str(tmp_path / "o.txt")
    ref = reference_output(f"pairwise_unaligned/{mode}", [mode] + flags + ["-q", q, "-d", d, "-f", "0", "-p", "8", "--quiet"])
    r = subprocess.run([CLI, mode] + flags + ["-q", q, "-d", d, "-f", "0", "-o", ours, "-p", "8"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = open(ours).read()
    assert text_digest(got) == ref
    assert got.count("***** No hits found *****") > 20
    if mode == "blastx":
        assert got.count(" Frame = -") > 50 and sum(got.count(f" Frame = {k}\n") for k in (1, 2, 3)) > 50


def test_vectorised_translation_equals_per_read_translation():
    """api.translate_codes (bench.py --config c3: 10^5 reads of one length) against api.translate_reads, incl. the ORF masking."""
    import numpy as np
    from diamond_b200 import api, synth
    w = synth.c3_workload(1500, 2000, 3)
    reads = ["".join("ACGT"[x] for x in row) for row in w["dna_codes"]]
    a, b = api.translate_reads(reads), api.translate_codes(w["dna_codes"])
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert (b[0] == 23).any() and (b[0] == 24).any()


# ---- frameshift alignment mode (blastx -F 15): the reference's legacy extension pipeline (align/legacy/*) over the 3-frame banded DP
# (dp/swipe/banded_3frame_swipe.cpp); goldens bx.xf / bx.xf0 / bx.xf3 = the unmodified reference with -F 15
XF_FIELDS = XT_FIELDS + ["qframe"]


@pytest.mark.parametrize("lvl,flags,ext", [("xf", ["--fast", "-f", "6"] + XF_FIELDS, "tsv"), ("xf0", ["--fast", "-f", "0"], "txt"), ("xf3", ["--sensitive"], "tsv"), ("xl", ["--long-reads"], "tsv")])
def test_blastx_frameshift_cli(oracle_lib, tmp_path, lvl, flags, ext):
    """Transcripts with \\ and / frameshift marks (cigar, btop, gapped sequences), begin and end of an alignment in different frames,
    the pairwise format with its "No hits found" record for EVERY unaligned read, and a many-shape mode (no gapped filter in the legacy pipeline)."""
    q, d = _files(_bx(), tmp_path)
    o = str(tmp_path / "o.out")
    r = subprocess.run([CLI, "blastx"] + flags + ([] if lvl == "xl" else ["-F", "15"]) + ["-q", q, "-d", d, "-o", o, "-p", "8", "--log"], capture_output=True, text=True)  # xl: --long-reads = --range-culling --top 10 -F 15
    assert r.returncode == 0, r.stderr
    assert open(o).read() == open(os.path.join(GOLDEN, f"bx.{lvl}.{ext}")).read()
    gold = json.load(open(os.path.join(GOLDEN, f"bx.{lvl}.counters.json")))
    log = r.stderr + r.stdout
    assert f"Target hits (stage 0) = {gold['targets']}" in log            # targets with a positive ungapped hit (QueryMapper::count_targets)
    assert f"Target hits (stage 3) = {gold['targets_stage2']}" in log     # targets that enter the traceback DP (the reference's TARGET_HITS2)


def test_blastx_frameshift_library(oracle_lib):
    """Through the C ABI: frame_shift in dmnd_search_opts, the end frame of an alignment in dmnd_match.reserved."""
    from diamond_b200 import api
    w = _bx()
    ql, qo = api.translate_reads(w["dna"], frame_shift=15)
    q_raw, q_lim = api.block_image(ql, qo)
    r_raw, r_lim = api.block_image(w["db_letters"], w["db_off"])
    g = api.Context(lib=oracle_lib, masking=1, motif_masking=1, query_contexts=6, frame_shift=15)
    m, tr, st = g.blastp(q_raw, q_lim, r_raw, r_lim)
    g.close()
    gold = ["\t".join(l.split("\t")[:12]) for l in open(os.path.join(GOLDEN, "bx.xf.tsv")).read().splitlines()]
    assert api.fmt6_translated(m, [len(r) for r in w["dna"]]).splitlines() == gold
    shifted = sum(1 for x in m if int(x["reserved"]) - 1 != int(x["query"]) % 6)
    assert shifted > 20 and (m["reserved"] > 0).all()  # alignments that end in another frame than they begin in
    fs_bytes = np.isin(tr, [0x41, 0x42]).sum()
    assert fs_bytes >= shifted


def test_frameshift_needs_translated_queries(oracle_lib):
    from diamond_b200 import api
    with pytest.raises(api.DmndError):
        g = api.Context(lib=oracle_lib, query_contexts=1, frame_shift=15)
        w = _bx()
        r_raw, r_lim = api.block_image(w["db_letters"], w["db_off"])
        g.blastp(r_raw, r_lim, r_raw, r_lim)


def test_blastx_frameshift_lanes(oracle_lib, monkeypatch):
    """The frameshift pipeline with three query lanes (each lane runs its own legacy rounds on its context): same output."""
    from diamond_b200 import api
    monkeypatch.setenv("DMND_LANES", "3")
    w = _bx()
    ql, qo = api.translate_reads(w["dna"], frame_shift=15)
    q_raw, q_lim = api.block_image(ql, qo)
    r_raw, r_lim = api.block_image(w["db_letters"], w["db_off"])
    g = api.Context(lib=oracle_lib, masking=1, motif_masking=1, query_contexts=6, frame_shift=15)
    m, _, _ = g.blastp(q_raw, q_lim, r_raw, r_lim)
    g.close()
    gold = ["\t".join(l.split("\t")[:12]) for l in open(os.path.join(GOLDEN, "bx.xf.tsv")).read().splitlines()]
    assert api.fmt6_translated(m, [len(r) for r in w["dna"]]).splitlines() == gold


def test_frameshift_repeated_calls_on_one_context(oracle_lib):
    """The P layer keeps its per-query states between calls (no page faults in steady state): a second frameshift search on the same
    context, over a different reference block, must not see the first one's match lists (regression: stale list pointers gave
    later blocks of a -b run matches of the wrong queries)."""
    from diamond_b200 import api
    w = _bx()
    ql, qo = api.translate_reads(w["dna"], frame_shift=15)
    q_raw, q_lim = api.block_image(ql, qo)
    nd = len(w["db_off"]) - 1
    half = nd // 2
    blocks = [api.block_image(w["db_letters"][: w["db_off"][half]], w["db_off"][: half + 1]),
              api.block_image(w["db_letters"][w["db_off"][half]:], w["db_off"][half:] - w["db_off"][half])]
    lens = [len(r) for r in w["dna"]]
    outs = []
    g = api.Context(lib=oracle_lib, masking=1, motif_masking=1, query_contexts=6, frame_shift=15)
    for r_raw, r_lim in blocks + blocks[:1]:
        m, _, _ = g.blastp(q_raw, q_lim, r_raw, r_lim)
        outs.append(api.fmt6_translated(m, lens))
    g.close()
    assert outs[0] == outs[2] and outs[0] != outs[1]
    for k, (r_raw, r_lim) in enumerate(blocks):  # each against a fresh context
        f = api.Context(lib=oracle_lib, masking=1, motif_masking=1, query_contexts=6, frame_shift=15)
        m, _, _ = f.blastp(q_raw, q_lim, r_raw, r_lim)
        f.close()
        assert api.fmt6_translated(m, lens) == outs[k]


def test_frameshift_with_reference_blocks_matches_the_reference(oracle_lib, tmp_path):
    """blastx -F 15 -b: per-block legacy runs joined per query; the reference re-derives the statistics of a joined record from its
    transcript (HspContext::parse), so `length` counts the frameshift marks there -- compared with the reference's file."""
    q, d = _files(_bx(), tmp_path)
    fields = "qseqid sseqid pident length mismatch gapopen qstart qend sstart send evalue bitscore cigar btop gaps nident qframe".split()
    for flags in (["--fast", "-b0.0002", "-f", "6"] + fields,):  # (--sensitive -b0.0001 -k 5 compared by hand: identical)
        o2 = str(tmp_path / "our.tsv")
        ref = reference_output("frameshift_blocks/" + " ".join(flags[:2]), ["blastx", "-q", q, "-d", d, "-F", "15", "-p", "8", "--quiet"] + flags)
        r = subprocess.run([CLI, "blastx", "-q", q, "-d", d, "-F", "15", "-p", "8", "-o", o2] + flags, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert text_digest(open(o2).read()) == ref


def test_frameshift_score_only_int16_overflow(oracle_lib, tmp_path):
    """A 40 kb read against 32 near-identical 13 500-letter targets: more than -k targets, so the score-only round runs, and every score
    (~79 000) saturates the reference's int16 SIMD lanes -- it repeats such a target alone, in its own band, in int32
    (dp/swipe/banded_3frame_swipe.cpp:600-607); host/legacy.inc does the same.  Compared with the reference's file."""
    from diamond_b200 import synth
    rng = np.random.default_rng(7)
    aa = "ARNDCQEGHILKMFPSTWYV"
    L = 13500
    prot = rng.integers(0, 20, L)
    q, d, o2 = (str(tmp_path / x) for x in ("q.fna", "d.faa", "our.tsv"))
    open(q, "w").write(">long\n" + "".join(synth._CODONS[aa[a]][0] for a in prot) + "\n")
    with open(d, "w") as f:
        for k in range(32):
            p = prot.copy()
            m = rng.random(L) < 0.002 * k
            p[m] = rng.integers(0, 20, int(m.sum()))
            f.write(f">t{k}\n" + "".join(aa[a] for a in p) + "\n")
        for k in range(200):
            f.write(f">r{k}\n" + "".join(aa[a] for a in rng.integers(0, 20, 300)) + "\n")
    want = reference_output("frameshift_int16_overflow", ["blastx", "--fast", "-q", q, "-d", d, "-F", "15", "-p", "8", "--quiet"])
    r = subprocess.run([CLI, "blastx", "--fast", "-q", q, "-d", d, "-F", "15", "-p", "8", "-o", o2], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = open(o2).read()
    assert text_digest(got) == want and len(got.splitlines()) == 25 and float(got.splitlines()[0].split("\t")[11]) > 30000  # raw score ~ 79 000 > 65 535
