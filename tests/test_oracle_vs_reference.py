"""Pins the oracle (oracle/dmnd_oracle.c under the host pipeline) against the REFERENCE ITSELF:
 * byte-identical fmt-6 output and equal --log stage counters with the committed golden fixtures, which were produced
   by running the unmodified reference (tests/golden/make_golden.py);
 * the reference's output on a further seed (tests/golden/reference_outputs.json, recorded by running it: conftest.reference_output).
CPU only."""
import json, os, subprocess, tempfile
import numpy as np
import pytest
from conftest import GOLDEN, reference_output, text_digest, workload_blocks


@pytest.mark.parametrize("name", ["c1", "fam2", "edge", "long"])  # "long": round-2 problems above max_swipe_dp (statistics passes)
@pytest.mark.parametrize("level,cbs", [("l0", 0), ("l1", 1)])
def test_fmt6_and_counters_match_reference_golden(oracle_lib, name, level, cbs):
    from diamond_b200 import api
    w, q_raw, q_lim, r_raw, r_lim = workload_blocks(name)
    ctx = api.Context(oracle_lib, threads=8, comp_based_stats=cbs)
    assert ctx.backend() == "oracle-cpu"
    m, _, st = ctx.blastp(q_raw, q_lim, r_raw, r_lim)
    ctx.close()
    gold = open(os.path.join(GOLDEN, f"{name}.{level}.tsv")).read()
    assert api.fmt6(m) == gold
    cn = json.load(open(os.path.join(GOLDEN, f"{name}.{level}.counters.json")))
    for k in ("seeds_hit", "seed_hits", "tentative_matches1", "tentative_matches2", "tentative_matches3"):
        assert st["seed"][k] == cn[k], k
    assert st["targets"] == cn["targets"]
    assert st["dp_problems_round2"] == cn["targets_round2"]
    assert ctx.params.seedp_bits == cn["seedp_bits"]


@pytest.mark.parametrize("seed", [101])
def test_live_reference_run(oracle_lib, seed):
    from diamond_b200 import api, synth
    w = synth.workload(300, 3000, seed)
    q_raw, q_lim = api.block_image(w["q_letters"], w["q_off"])
    r_raw, r_lim = api.block_image(w["db_letters"], w["db_off"])
    with tempfile.TemporaryDirectory() as td:
        q, d = (os.path.join(td, x) for x in ("q.faa", "d.faa"))
        synth.write_fasta(q, w["q_letters"], w["q_off"], "q")
        synth.write_fasta(d, w["db_letters"], w["db_off"], "d")
        gold = reference_output(f"live_reference_run/{seed}", ["blastp", "--fast", "-q", q, "-d", d, "-f", "6", "-p", "8", "--masking", "0",
                                                                "--motif-masking", "0", "--quiet"])
    ctx = api.Context(oracle_lib, threads=8, comp_based_stats=1)
    m, _, _ = ctx.blastp(q_raw, q_lim, r_raw, r_lim)
    ctx.close()
    assert text_digest(api.fmt6(m)) == gold


@pytest.mark.parametrize("lanes", ["1", "3", "3-nofuse"])
def test_query_lanes_do_not_change_results(oracle_lib, lanes, monkeypatch):
    """The P layer may split the query block into lanes that run concurrently: output must be independent of it.  "3-nofuse" =
    DMND_NO_FUSE, which also turns the device bridge off: single-shape blastp then takes the host path in every lane."""
    from diamond_b200 import api
    monkeypatch.setenv("DMND_LANES", lanes[0])
    if lanes.endswith("nofuse"):
        monkeypatch.setenv("DMND_NO_FUSE", "1")
    w, q_raw, q_lim, r_raw, r_lim = workload_blocks("fam2")
    ctx = api.Context(oracle_lib, threads=8, comp_based_stats=1, want_transcript=True)
    m, tr, st = ctx.blastp(q_raw, q_lim, r_raw, r_lim)
    ctx.close()
    assert api.fmt6(m) == open(os.path.join(GOLDEN, "fam2.l1.tsv")).read()
    cn = json.load(open(os.path.join(GOLDEN, "fam2.l1.counters.json")))
    assert st["seed"]["tentative_matches3"] == cn["tentative_matches3"] and st["seed"]["seeds_hit"] >= cn["seeds_hit"]
    assert np.all(m["transcript_off"] + m["transcript_len"] <= len(tr)) and np.array_equal(m["transcript_len"], m["length"])
    ops = np.concatenate([tr[a:a + n] for a, n in zip(m["transcript_off"][:50], m["transcript_len"][:50])]) >> 6
    assert set(np.unique(ops)) <= {0, 1, 2, 3}


def test_evalue_within_tolerance_of_printed_reference_values(oracle_lib):
    """north_star: e-values within 1e-6 relative.  The reference prints %.2e, so compare at that precision and make
    sure no value sits on a rounding edge by also checking the raw double against the printed one to 0.5 % (3 digits)."""
    from diamond_b200 import api
    w, q_raw, q_lim, r_raw, r_lim = workload_blocks("c1")
    ctx = api.Context(oracle_lib, threads=8, comp_based_stats=1)
    m, _, _ = ctx.blastp(q_raw, q_lim, r_raw, r_lim)
    ctx.close()
    gold = [l.split("\t") for l in open(os.path.join(GOLDEN, "c1.l1.tsv")).read().splitlines()]
    assert len(gold) == len(m)
    for g, x in zip(gold, m):
        ref = float(g[10])
        if ref > 0:
            assert abs(x["evalue"] - ref) / ref < 5.1e-3
        assert ("0.0" if x["evalue"] == 0 else "%.2e" % x["evalue"]) == g[10]


def test_cli_rejects_what_it_does_not_implement(oracle_lib):
    from conftest import ROOT
    cli = os.path.join(ROOT, "oracle", "_build", "dmnd-oracle-cli")
    r = subprocess.run([cli, "blastp", "-q", "x", "-d", "y", "-o", "z", "--masking", "seg"], capture_output=True, text=True)
    assert r.returncode != 0 and "masking" in r.stderr
    r = subprocess.run([cli, "blastp", "-q", "x", "-d", "y", "-o", "z", "--faster"], capture_output=True, text=True)
    assert r.returncode != 0 and "unsupported option" in r.stderr
    r = subprocess.run([cli, "blastx"], capture_output=True, text=True)
    assert r.returncode != 0


@pytest.mark.parametrize("name", ["c1", "edge", "long"])
def test_fused_rounds_equal_two_round_execution(oracle_lib, name, monkeypatch):
    """Queries with few targets answer round 2 from the traceback results of their round-1 problems (pipeline.cpp,
    Driver::start); DMND_NO_FUSE=1 runs the reference's two separate rounds.  Same matches, same problem and cell counts."""
    from diamond_b200 import api
    w, q_raw, q_lim, r_raw, r_lim = workload_blocks(name)
    out = []
    for no_fuse in (False, True):
        if no_fuse:
            monkeypatch.setenv("DMND_NO_FUSE", "1")
        else:
            monkeypatch.delenv("DMND_NO_FUSE", raising=False)
        ctx = api.Context(oracle_lib, threads=8, comp_based_stats=1, want_transcript=(name != "long"))
        m, tr, st = ctx.blastp(q_raw, q_lim, r_raw, r_lim)
        ctx.close()
        out.append((api.fmt6(m), m.copy(), tr.copy(), st))
    assert out[0][0] == out[1][0]
    for f in ("dp_problems_round1", "dp_problems_round2", "cells_round1", "cells_round2", "matches", "queries_aligned"):
        assert out[0][3][f] == out[1][3][f], f
    for a, b in zip(out[0][1], out[1][1]):
        assert np.array_equal(out[0][2][a["transcript_off"]: a["transcript_off"] + a["transcript_len"]],
                              out[1][2][b["transcript_off"]: b["transcript_off"] + b["transcript_len"]])
