"""SURVEY 8(f) rank 1, first half: the reference's DEFAULT sensitivity (`diamond blastp` without --fast: two shapes of
weight 10, entropy cut 0.8, stage-2 ungapped window filter with the e-value 10 000 cutoff table, search/setup.cpp:43-47,
:90-93; search/stage2.h:41-154; dp/ungapped_simd.cpp:32-88) in the oracle and the host pipeline, pinned against the
S1 goldens (the reference run with no sensitivity flag and its default masking) and a live run on real proteins.  CPU only."""
import ctypes as C, json, os, re, subprocess
import numpy as np
import pytest
from conftest import GOLDEN, ROOT, reference_output, text_digest, workload_blocks

NR10K = os.path.join(GOLDEN, "refdata", "nr_10k.faa.gz")  # a sample of the reference's nr_10k.faa


@pytest.mark.parametrize("name", ["c1", "fam2", "edge", "long", "rep"])
def test_default_sensitivity_matches_reference_golden(oracle_lib, name):
    from diamond_b200 import api
    w, q_raw, q_lim, r_raw, r_lim = workload_blocks(name)
    ctx = api.Context(oracle_lib, threads=8, comp_based_stats=1, masking=1, motif_masking=1, sensitivity=1)
    assert ctx.params.n_shapes == 2 and ctx.params.shape_weight == 10 and ctx.params.ungapped_evalue == 10000.0
    m, _, st = ctx.blastp(q_raw, q_lim, r_raw, r_lim)
    ctx.close()
    assert api.fmt6(m) == open(os.path.join(GOLDEN, f"{name}.s1.tsv")).read()
    cn = json.load(open(os.path.join(GOLDEN, f"{name}.s1.counters.json")))
    for k in ("seeds_hit", "seed_hits", "tentative_matches1", "tentative_matches2", "tentative_matches3"):
        assert st["seed"][k] == cn[k], k  # summed over both shapes, like the reference's statistics
    assert st["targets"] == cn["targets"] and st["dp_problems_round2"] == cn["targets_round2"] and ctx.params.seedp_bits == cn["seedp_bits"]


@pytest.mark.parametrize("name", ["c1", "edge", "rep"])  # (fam2.s2 is pinned too, but takes the scalar oracle half a minute)
def test_mid_sensitive_matches_reference_golden(oracle_lib, name):
    """--mid-sensitive: 8 shapes of weight 9 (search/setup.cpp:201-210), entropy cut 1.0, the same stage-2 window filter."""
    from diamond_b200 import api
    w, q_raw, q_lim, r_raw, r_lim = workload_blocks(name)
    ctx = api.Context(oracle_lib, threads=8, comp_based_stats=1, masking=1, motif_masking=1, sensitivity=2)
    assert ctx.params.n_shapes == 8 and ctx.params.shape_weight == 9
    m, _, st = ctx.blastp(q_raw, q_lim, r_raw, r_lim)
    ctx.close()
    assert api.fmt6(m) == open(os.path.join(GOLDEN, f"{name}.s2.tsv")).read()
    cn = json.load(open(os.path.join(GOLDEN, f"{name}.s2.counters.json")))
    for k in ("seeds_hit", "seed_hits", "tentative_matches1", "tentative_matches2", "tentative_matches3"):
        assert st["seed"][k] == cn[k], k
    assert st["targets"] == cn["targets"] and st["dp_problems_round2"] == cn["targets_round2"]


@pytest.mark.parametrize("name", ["c1", "edge", "long", "rep"])  # (fam2.s3: 2 x 10^7 stage-0 pairs, two minutes in the scalar oracle; run it by hand)
def test_sensitive_matches_reference_golden(oracle_lib, name):
    """--sensitive: 16 shapes of weight 8 (search/setup.cpp:94-110) and the gapped filter (align/gapped_filter.cpp:33-63: 64- and
    128-diagonal scans of the int8 query profile, dp/scan_diags.cpp, cutoffs from CutoffTable2D at e-values 2000 and 1)."""
    from diamond_b200 import api
    w, q_raw, q_lim, r_raw, r_lim = workload_blocks(name)
    ctx = api.Context(oracle_lib, threads=8, comp_based_stats=1, masking=1, motif_masking=1, sensitivity=3)
    p = ctx.params
    assert p.n_shapes == 16 and p.shape_weight == 8 and p.gapped_filter_evalue == 1.0
    assert 10 < p.gapped_cutoff1[9][9] < p.gapped_cutoff2[9][9] < 200  # the second stage (e-value 1) is the stricter one
    m, _, st = ctx.blastp(q_raw, q_lim, r_raw, r_lim)
    ctx.close()
    assert api.fmt6(m) == open(os.path.join(GOLDEN, f"{name}.s3.tsv")).read()
    cn = json.load(open(os.path.join(GOLDEN, f"{name}.s3.counters.json")))
    for k in ("seeds_hit", "seed_hits", "tentative_matches1", "tentative_matches2", "tentative_matches3"):
        assert st["seed"][k] == cn[k], k
    assert st["targets"] == cn["targets"] and st["dp_problems_round2"] == cn["targets_round2"]
    assert st["targets_extended"] == cn["targets_extended"], "targets that survive the gapped filter (Target hits (stage 3))"
    if name == "c1":
        assert st["targets_extended"] < st["targets"]  # the filter does remove targets here


@pytest.mark.parametrize("sens,level,name", [(4, "s4", "edge"), (5, "s5", "c1"), (5, "s5", "edge"), (6, "s6", "edge")])  # (c1 / rep goldens of all three exist; the scalar oracle needs a minute for c1.s6)
def test_more_very_ultra_sensitive_match_reference_golden(oracle_lib, name, sens, level):
    """--more-sensitive (the 16 shapes of --sensitive, no motif masking, BANDED_SLOW bands), --very-sensitive (14 shapes of weight 7,
    Hamming cutoff 9, one index chunk, ungapped e-value 10^5) and --ultra-sensitive (64 shapes, 3 x 10^5): sensitivity_traits
    (search/setup.cpp:40-54), shape_codes (:111-200), Extension::band (align/gapped_score.cpp:41-72)."""
    from diamond_b200 import api
    w, q_raw, q_lim, r_raw, r_lim = workload_blocks(name)
    assert oracle_lib.dmnd_mode_motif_masking(sens) == 0 and oracle_lib.dmnd_mode_motif_masking(3) == 1
    ctx = api.Context(oracle_lib, threads=8, comp_based_stats=1, masking=1, motif_masking=0, sensitivity=sens)
    p = ctx.params
    assert (p.n_shapes, p.shape_weight, p.hamming_id, p.index_chunks) == {4: (16, 8, 11, 4), 5: (14, 7, 9, 1), 6: (64, 7, 9, 1)}[sens]
    m, _, st = ctx.blastp(q_raw, q_lim, r_raw, r_lim)
    ctx.close()
    assert api.fmt6(m) == open(os.path.join(GOLDEN, f"{name}.{level}.tsv")).read()
    cn = json.load(open(os.path.join(GOLDEN, f"{name}.{level}.counters.json")))
    for k in ("seeds_hit", "seed_hits", "tentative_matches1", "tentative_matches2", "tentative_matches3"):
        assert st["seed"][k] == cn[k], k
    assert st["targets"] == cn["targets"] and st["targets_extended"] == cn["targets_extended"] and st["dp_problems_round2"] == cn["targets_round2"]


def test_ungapped_cutoffs_and_hit_scores(oracle_lib):
    """The hit score is the ungapped window score (search/stage2.h:144-147): above the cutoff of the query's length class,
    at most 255 where the reference's int8 kernel scored the call (>= 4 survivors), unbounded for the scalar calls; the
    many-target workload must contain both kinds, or the call-size rule is not exercised."""
    from diamond_b200 import api
    w, q_raw, q_lim, r_raw, r_lim = workload_blocks("fam2")
    ctx = api.Context(oracle_lib, threads=8, masking=0, motif_masking=0, sensitivity=1)
    p = ctx.params
    cut = list(p.ungapped_cutoff)
    assert cut[0] == 0 and all(cut[b] <= cut[b + 1] for b in range(1, 31)) and 20 < cut[9] < 60 and p.short_query_ungapped_cutoff > 0
    qb, rb = ctx.upload(q_raw, q_lim), ctx.upload(r_raw, r_lim)
    scores = []
    for sid in (0, 1):
        hits, cn = ctx.search_shape(qb, rb, sid)
        assert cn["tentative_matches2"] <= cn["tentative_matches1"] and cn["tentative_matches3"] == len(hits)
        sc = (hits["subject_score"] >> np.uint64(48)).astype(np.int64)
        qlen = (np.diff(q_lim) - 1)[hits["query"]]
        cutoff = np.where(qlen <= p.short_query_max_len, p.short_query_ungapped_cutoff, np.array(cut)[np.floor(np.log2(qlen)).astype(int) + 1])
        assert np.all(sc > cutoff)
        scores.append(sc)
    ctx.free_block(qb); ctx.free_block(rb); ctx.close()
    sc = np.concatenate(scores)
    assert (sc == 255).sum() > 100 and (sc > 255).sum() > 0 and (sc < 255).sum() > 100


def test_live_reference_default_sensitivity_on_real_proteins(tmp_path):
    import gzip
    cli = os.path.join(ROOT, "oracle", "_build", "dmnd-oracle-cli")
    sub = tmp_path / "nr.faa"
    sub.write_bytes(gzip.open(NR10K).read())
    our_out = tmp_path / "our.tsv"
    pats = (r"Seeds hit\s+= (\d+)", r"Hits \(filter stage 0\) = (\d+)", r"Hits \(filter stage 1\) = (\d+)", r"Hits \(filter stage 2\) = (\d+)", r"Hits \(filter stage 3\) = (\d+)")
    ref = reference_output("real_proteins/default", ["blastp", "-q", str(sub), "-d", str(sub), "-f", "6", "-p", "8", "--log"], pats)
    o = subprocess.run([cli, "blastp", "-q", str(sub), "-d", str(sub), "-o", str(our_out), "-p", "8", "--log"], capture_output=True, text=True, check=True)
    assert text_digest(our_out.read_text(), o.stdout + o.stderr, pats) == ref and ref["bytes"] > 10000
