"""Writes tests/golden/refdata/: a sample of the reference's own test inputs (its src/test directory) and the command lines of
its regression tests (CMakeLists.txt), so that the tests replaying them need nothing outside this repository.

    python tests/golden/make_refdata.py REFERENCE_CHECKOUT   # needs oracle/_ref/diamond (make ref)
    DMND_RECORD_REFERENCE=1 python -m pytest tests -m "not gpu"   # then record the reference's outputs on these inputs (make ref)

Kept whole: 1.faa .. 4.faa and data.faa (300 proteins).  Sampled, under the same names: the 12 shortest reads with an alignment among the first
200 nanopore reads (SRR14011045_1.fna.gz; the first 3 of them in SRR14011045_1.fastq), the first 20 proteins of nr_300.faa, and of
nr_10k.faa the first 30 proteins plus every target the reference's committed blastx-nanopore.out reports for the sampled reads
and every target its committed blastp-daa.out archive holds for the sampled nr_300 proteins.  test.daa (stored gzip-compressed) is the
reference's -f 100 archive of the blastp-daa case on these inputs (its makedb of the sampled nr_10k.faa, then that case's command
line), the DAA file the view case reads."""
import gzip, json, os, re, shlex, shutil, subprocess, sys, tempfile

REF = sys.argv[1] if len(sys.argv) > 1 else "."
TD = os.path.join(REF, "src", "test")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "refdata")
REF_BIN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", "oracle", "_ref", "diamond")
NANO_READS, FASTQ_READS, NR300, NR10K_HEAD = 12, 3, 20, 30
# the cases this repository's CLI covers; the others need options outside it (taxonomy, BLAST databases, --max-hsps 0, matrix
# adjustment (--comp-based-stats 2-4), other matrices, --global-ranking, linclust / realign)
CASES = ["blastp", "blastp-mid-sens", "blastp-f0", "blastx-nanopore", "blastx-nanopore-fna",
         "diamond-test-blastp-default", "diamond-test-blastp-multithreaded", "diamond-test-blastp-more-sensitive",
         "diamond-test-blastp-very-sensitive", "diamond-test-blastp-ultra-sensitive", "diamond-test-blastp-target-parallel",
         "diamond-test-blastp-query-indexed", "diamond-test-blastp-comp-based-stats-0", "diamond-test-blastp-target-seqs",
         "diamond-test-blastp-evalue", "diamond-test-blastp-pairwise-format", "diamond-test-blastp-paf-format", "diamond-test-blastp-top",
         "blastp-blocked", "diamond-test-blastp-blocked",  # -b: reference blocks + join_blocks
         "view",        # a DAA file of the reference read back (`view -a test.daa`)
         "blastp-daa"]  # -f 100: the reference's archive, byte for byte


def records(text, mark):
    recs, cur = [], []
    for line in text.splitlines(keepends=True):
        if line.startswith(mark) and cur and (mark == ">" or len(cur) == 4):
            recs.append("".join(cur)); cur = []
        cur.append(line)
    if cur:
        recs.append("".join(cur))
    return recs


def save(name, text, gz=True):
    data = text.encode()
    if gz:
        with gzip.GzipFile(os.path.join(OUT, name + ".gz"), "wb", mtime=0) as f:
            f.write(data)
    else:
        open(os.path.join(OUT, name), "wb").write(data)


def main():
    os.makedirs(OUT, exist_ok=True)
    for f in ("1.faa", "2.faa", "3.faa", "4.faa"):
        save(f, open(os.path.join(TD, f)).read(), gz=False)
    save("data.faa", open(os.path.join(TD, "data.faa")).read())
    fq = records(open(os.path.join(TD, "SRR14011045_1.fastq")).read(), "@")[:200]
    aligned = {l.split("\t")[0] for l in open(os.path.join(TD, "blastx-nanopore.out"))}
    cand = [k for k in range(len(fq)) if fq[k].split()[0][1:] in aligned]
    pick = sorted(sorted(cand, key=lambda k: (len(fq[k]), k))[:NANO_READS])  # (quality lines compress poorly)
    save("SRR14011045_1.fastq", "".join(fq[k] for k in pick[:FASTQ_READS]))
    fna = records(gzip.open(os.path.join(TD, "SRR14011045_1.fna.gz")).read().decode(), ">")
    fna = [fna[k] for k in pick]
    with gzip.GzipFile(os.path.join(OUT, "SRR14011045_1.fna.gz"), "wb", mtime=0) as f:  # read gzip-compressed by the CLI itself
        f.write("".join(fna).encode())
    reads = {r.split()[0][1:] for r in fna}
    hit = {l.split("\t")[1] for l in open(os.path.join(TD, "blastx-nanopore.out")) if l.split("\t")[0] in reads}
    nr300 = records(open(os.path.join(TD, "nr_300.faa")).read(), ">")[:NR300]
    q300 = {r.split()[0][1:] for r in nr300}
    with tempfile.TemporaryDirectory() as tmp:
        shutil.copy(os.path.join(TD, "blastp-daa.out"), os.path.join(tmp, "a.daa"))  # (view reads NAME.daa)
        subprocess.run([REF_BIN, "view", "-a", os.path.join(tmp, "a.daa"), "-f", "6", "qseqid", "sseqid", "-o", os.path.join(tmp, "v"), "--quiet"], check=True)
        daa = open(os.path.join(tmp, "v")).read()
    hit |= {l.split("\t")[1] for l in daa.splitlines() if l.split("\t")[0] in q300}
    nr = records(open(os.path.join(TD, "nr_10k.faa")).read(), ">")
    save("nr_10k.faa", "".join(r for k, r in enumerate(nr) if k < NR10K_HEAD or r.split()[0][1:] in hit))
    save("nr_300.faa", "".join(nr300))
    txt = open(os.path.join(REF, "CMakeLists.txt")).read()
    cmds = {m.group(1): m.group(2) for m in re.finditer(r'-DNAME=(\S+) "-DARGS=([^"]*)"', txt)}
    cmds.update({m.group(1): m.group(2) for m in re.finditer(r'add_diamond_test\((\S+) "([^"]*)"\)', txt)})
    with open(os.path.join(OUT, "ctest_commands.json"), "w") as f:
        json.dump({k: shlex.split(cmds[k]) for k in CASES}, f, indent=1)
        f.write("\n")
    with tempfile.TemporaryDirectory() as tmp:
        for f in ("nr_10k.faa", "nr_300.faa"):
            open(os.path.join(tmp, f), "wb").write(gzip.open(os.path.join(OUT, f + ".gz")).read())
        subprocess.run([REF_BIN, "makedb", "--in", os.path.join(tmp, "nr_10k.faa"), "-d", os.path.join(tmp, "nr_10k"), "--quiet"], check=True)
        args = [a.replace("${TD}", tmp) for a in shlex.split(cmds["blastp-daa"])]
        args = [os.path.join(tmp, a) if a == "nr_10k.dmnd" else a for a in args]
        subprocess.run([REF_BIN] + args + ["-o", os.path.join(tmp, "test.daa"), "--quiet"], check=True)
        with gzip.GzipFile(os.path.join(OUT, "test.daa.gz"), "wb", mtime=0) as f:
            f.write(open(os.path.join(tmp, "test.daa"), "rb").read())


if __name__ == "__main__":
    main()
