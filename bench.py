#!/usr/bin/env python
"""bench.py -- GCUPS of the seed-and-extend hot path (BASELINE.json metric) on N B200s of one node.

  python bench.py --gpus N --steps K --warmup W [--config c2|c3|c4|c5]   our arm (CUDA library behind the C ABI)
  python bench.py --impl reference --gpus N --steps K ...               the UNMODIFIED reference (oracle/_ref/diamond) on host cores

One "step" = one full pass of the hot path (masked blocks -> seed search stages 0-2 -> extension rounds 1+2 -> culling) over
one batch of synthetic queries against the resident reference block.  Configurations (BASELINE.json `configs`, SURVEY 8):
  c2 (default, the configuration the metric is quoted on): blastp --fast, 1 M queries (len <= 300) x 100 k-protein DB
  c3: blastx --fast, 100 k DNA reads of 150 nt (six translated frames each) x 100 k-protein DB
  c4: blastp --sensitive, 1 M queries x 500 k-protein DB (16 shapes, gapped filter)
  c5: blastx --very-sensitive -F 15 (frameshift alignment: legacy pipeline + 3-frame banded DP, every alignment traced back), 12 500 reads of
      600 nt with single-nucleotide indels (the per-GPU share of configs[4]'s 100 k queries on 8 GPUs) x 1 M-protein DB; cells = 3 x band x cols
At N > 1 every rank processes its own query block against the same DB (query sharding, no data-path collective; the packed
reference block is NCCL-broadcast once) -> "weak".
GCUPS numerator = algorithmic DP cells = sum over every banded DP problem of rounds 1 and 2 of band x cols
(dp/dp.h:121-124); it is a property of the workload (the DP target list is parity-checked against the reference).
`value` times steps with both blocks already resident in HBM; `e2e` times dmnd_blastp() with pinned HOST buffers
(block upload, masking, problem lists, hit/result downloads inside).  Inputs exceed the 126 MB L2.
Flags: the reference's DEFAULTS (tantan masking of both blocks, motif soft masking, Hauser composition bias) on both arms.
Masking belongs to loading a block (run/double_indexed.cpp:122-127, :737-741): resident blocks are masked when they are
made resident (outside the `value` region, like the upload); `e2e` and the reference arm mask inside the timed region.

Reference arm: the stock CLI on the SAME configuration (all queries of rank 0's block, FASTA in, fmt 6 out, whole process wall
time), `-p` = the fastest of the thread counts tried on a 100 k-query sample; one process run per step, --steps steps (a full
run takes ~10 s).  The cell count of the configuration comes from profiles/workload_cells.json, or from the table --cells-json
names (`--emit-cells` or a run of our arm writes it there; commit the entry to profiles/workload_cells.json to keep it): the
reference process never loads the CUDA library.
"""
import argparse, json, os, subprocess, sys, tempfile, threading, time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "diamond")
CELLS_JSON = os.path.join(ROOT, "profiles", "workload_cells.json")
DUMP_MAX_ROWS = 1 << 18  # 17 match fields + the row index, float64: 38 MB at most
DUMP_MAX_TRANSCRIPT = 1 << 22  # edit-transcript bytes of the sampled rows, float32: 16 MB at most
NO_MASKING = ["--masking", "0", "--motif-masking", "0"]  # parity-ladder rung L1 (SURVEY 8c); [] = the reference's default flags

CONFIGS = {
    "c2": dict(kind="blastp", sens=0, flag="--fast", queries=1_000_000, db=100_000, seed=2, label="BASELINE configs[1]",
               what="blastp --fast, {q} synthetic queries (len<=300) per GPU x {d}-protein DB"),
    "c3": dict(kind="blastx", sens=0, flag="--fast", queries=100_000, db=100_000, seed=3, label="BASELINE configs[2]",
               what="blastx --fast, {q} synthetic DNA reads (150 nt, six frames) per GPU x {d}-protein DB"),
    "c4": dict(kind="blastp", sens=3, flag="--sensitive", queries=1_000_000, db=500_000, seed=4, label="BASELINE configs[3]",
               what="blastp --sensitive, {q} synthetic queries (len<=300) per GPU x {d}-protein DB"),
    # configs[4]: "very-sensitive with frameshift + traceback": frameshift alignment exists for translated searches only (basic/config.cpp:822-823), so
    # the queries are DNA reads (600 nt, 70 % of them with a single-nucleotide insertion or deletion); every alignment is traced back in this mode
    "c5": dict(kind="blastx", sens=5, flag="--very-sensitive", frame_shift=15, read_len=600, indel=0.7, queries=12_500, db=1_000_000, seed=5, label="BASELINE configs[4] (per-GPU share of its 8-GPU layout: 100 000 reads / 8)",
               what="blastx --very-sensitive -F 15 (frameshift alignment, traceback), {q} synthetic DNA reads (600 nt, six frames) per GPU x {d}-protein DB"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--queries", type=int, default=None, help="queries (reads) per GPU; default: the configuration's")
    ap.add_argument("--db", type=int, default=None)
    ap.add_argument("--sample", type=int, default=100_000, help="queries of the bounded CPU-baseline sample of our arm")
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--emit-cells", default=None, help="comma list of reference thread counts: print the configuration's cell counts (and update --cells-json) and exit")
    ap.add_argument("--cells-json", default=None, help="cell-count table to read besides profiles/workload_cells.json, and to update with this run's count")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", help="write the matches of the last timed step as DIR/<field>.npy (float64; "
                    f"a fixed, seeded sample of at most {DUMP_MAX_ROWS} rows) and their edit transcripts, if any, as DIR/transcripts.npy")
    ap.add_argument("--masking", type=int, default=1, choices=[0, 1], help="1 = reference default flags (tantan + motif masking), 0 = --masking 0 --motif-masking 0 on both arms")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl == "reference" or a.emit_cells):
        ap.error("--dump-outputs writes what the timed CUDA path computed: not with --impl reference or --emit-cells")
    c = CONFIGS[a.config]
    a.queries = a.queries or c["queries"]; a.db = a.db or c["db"]; a.seed = c["seed"] if a.seed is None else a.seed
    return a


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.p, self.index = [], None, index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                      stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: [self.rows.append(l) for l in self.p.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def mark(self):
        """Row count now: the timed region's samples are the rows between two marks (the sampler process is started BEFORE the warm-up:
        its NVML initialisation stalls kernel launches for ~100 ms and must not fall into the timed region)."""
        return len(self.rows)

    def stop(self, first=0, last=None):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        for l in self.rows[first:last]:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v == "Active":
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def effective_cpus():
    """min(visible CPUs, cgroup CFS quota): what 'all the host threads it can use' means inside a quota-limited container."""
    n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, -(-int(q) // int(per))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, -(-q // per)))
        except Exception:
            pass
    return n


def make_workload(args, rank, n=None):
    """The rank's synthetic blocks.  Returns a dict: q_raw/q_lim/r_raw/r_lim (block images), ctx (Context keyword arguments), and
    what the reference arm needs to write its FASTA files."""
    from diamond_b200 import api, synth
    c = CONFIGS[args.config]
    n = n or args.queries
    if c["kind"] == "blastx":
        fs = c.get("frame_shift", 0)
        w = synth.c3_workload(args.queries, args.db, args.seed, read_len=c.get("read_len", 150), q_stream=rank, indel_rate=c.get("indel", 0.0))
        codes = w["dna_codes"][:n]
        ql, qo = api.translate_codes(codes, frame_shift=fs)
        q_raw, q_lim = api.block_image(ql, qo)
        out = {"dna_codes": codes, "read_lens": [codes.shape[1]] * n, "ctx": dict(sensitivity=c["sens"], query_contexts=6, frame_shift=fs)}
    else:
        w = synth.workload(args.queries, args.db, args.seed, q_stream=rank)
        q_raw, q_lim = api.block_image(w["q_letters"][: w["q_off"][n]], w["q_off"][: n + 1])
        out = {"q_letters": w["q_letters"][: w["q_off"][n]], "q_off": w["q_off"][: n + 1], "ctx": dict(sensitivity=c["sens"])}
    r_raw, r_lim = api.block_image(w["db_letters"], w["db_off"])
    out.update(q_raw=q_raw, q_lim=q_lim, r_raw=r_raw, r_lim=r_lim, db_letters=w["db_letters"], db_off=w["db_off"], n=n)
    return out


def write_fasta(wl, n, td):
    """First n queries of the workload + the whole DB as FASTA."""
    from diamond_b200 import synth
    d = os.path.join(td, "d.faa")
    synth.write_fasta(d, wl["db_letters"], wl["db_off"], "d")
    if "dna_codes" in wl:
        q = os.path.join(td, "q.fna")
        synth.write_dna_codes_fasta(q, wl["dna_codes"][:n])
    else:
        q = os.path.join(td, "q.faa")
        synth.write_fasta(q, wl["q_letters"][: wl["q_off"][n]], wl["q_off"][: n + 1], "q")
    return q, d


def run_reference(args, q, d, out, threads):
    c = CONFIGS[args.config]
    cmd = [REF_BIN, c["kind"], c["flag"], "-q", q, "-d", d, "-f", "6", "-o", out, "-p", str(threads), "--log"] + ([] if args.masking else NO_MASKING)
    if c.get("frame_shift"):
        cmd += ["-F", str(c["frame_shift"])]
    t0 = time.perf_counter()
    r = subprocess.run(cmd, capture_output=True, text=True)
    dt = time.perf_counter() - t0
    if r.returncode != 0:
        raise RuntimeError("reference failed: " + r.stderr[-400:])
    return dt


def fmt6_of(wl, m):
    from diamond_b200 import api
    return api.fmt6_translated(m, wl["read_lens"]) if "dna_codes" in wl else api.fmt6(m)


def cells_key(args, n, threads):
    return f"{args.config}:q{n}:db{args.db}:seed{args.seed}:masking{args.masking}:p{threads}:stream0"


def load_cells(extra=None):
    best = {}
    for p in (CELLS_JSON, extra):
        try:
            best.update(json.load(open(p)))
        except Exception:
            pass
    return best


def lookup_cells(args, n, threads):
    """(cells, note) of the first n queries of rank 0's block; the exact -p entry if there is one, else the entry of another thread
    count of the same configuration (the cell count moves by < 0.1 % with seedp_bits)."""
    tab = load_cells(args.cells_json)
    k = cells_key(args, n, threads)
    if k in tab:
        return tab[k], "cell count of this configuration from profiles/workload_cells.json (our arm, same -p)"
    pre = k.split(":p")[0]
    for kk, v in sorted(tab.items()):
        if kk.startswith(pre + ":p"):
            return v, f"cell count from profiles/workload_cells.json entry {kk} (no entry for -p {threads})"
    return None, ("no cached cell count for this configuration: run `python bench.py --emit-cells <threads> --cells-json FILE` on a B200 "
                  "and pass the same --cells-json here (or commit the entry to profiles/workload_cells.json)")


def sample_matches(m, tr):
    """The match fields of one step as float64 columns (every integer field is exact there): all rows, or a sorted sample of
    DUMP_MAX_ROWS row indices drawn with a fixed seed, so that two builds that return the same matches dump the same rows.
    Where the step returns edit transcripts, those of the sampled rows in row order (up to DUMP_MAX_TRANSCRIPT bytes) stand in for
    transcript_off: the offsets depend on how the library laid out its transcript buffer (its host thread count), not only on the
    results."""
    import numpy as np
    rows = np.arange(len(m))
    if len(m) > DUMP_MAX_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(len(m), DUMP_MAX_ROWS, replace=False))
    out = {name: m[name][rows].astype(np.float64) for name in m.dtype.names if not name.startswith("_") and name != "transcript_off"}
    out["row"] = rows.astype(np.float64)
    out["n_matches"] = np.array([len(m)], dtype=np.float64)
    if len(tr):
        parts, total = [], 0
        for off, n in zip(m["transcript_off"][rows], m["transcript_len"][rows]):
            if total + int(n) > DUMP_MAX_TRANSCRIPT:
                break
            parts.append(tr[int(off): int(off) + int(n)]); total += int(n)
        out["transcripts"] = (np.concatenate(parts) if parts else np.zeros(0, np.uint8)).astype(np.float32)
    return out


def dump_outputs(d, arrays):
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a)


_result_fd = None


def emit(obj):
    """stdout carries exactly ONE line, the JSON result: fd 1 is pointed at stderr for the run (NCCL's version banner and child
    processes print there) and the result goes to the saved descriptor."""
    os.write(_result_fd if _result_fd is not None else 1, (json.dumps(obj) + "\n").encode())


def main():
    global _result_fd
    args = parse()
    if args.gpus > 1 and "RANK" not in os.environ:
        # launched plainly with --gpus N: re-launch as one rank per GPU (what the driver does itself with torch.distributed.run)
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                                   "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29533"), os.path.abspath(__file__)] + sys.argv[1:])
    sys.stdout.flush()
    _result_fd = os.dup(1)
    os.dup2(2, 1)
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    ncpu = effective_cpus()
    ref_threads = ncpu  # seedp_bits follows -p (setup.cpp:306-309): both arms are run with the same value
    c = CONFIGS[args.config]
    config = {"workload": c["what"].format(q=args.queries, d=args.db) + f" ({c['label']})", "config": args.config,
              "queries_per_gpu": args.queries, "db_seqs": args.db, "parallelism": f"query-sharded x{world}", "seed": args.seed,
              "flags": f"{c['flag']} (reference defaults: tantan masking, motif masking, comp-based-stats 1) -k 25 -e 0.001" if args.masking else f"{c['flag']} --masking 0 --motif-masking 0 --comp-based-stats 1 -k 25 -e 0.001",
              "masking": "resident blocks are masked when made resident (block load); e2e and the reference arm mask inside the timed region" if args.masking else "off on both arms",
              "reference_threads": ref_threads, "visible_cpus": os.cpu_count(),
              "l2": "inputs (query + reference blocks, 100+ MB per GPU) larger than the 126 MB L2"}
    metric = f"GCUPS {c['kind']} {c['flag']}"

    if args.impl == "reference":
        if rank != 0:
            return
        if not os.path.exists(REF_BIN):
            emit({"impl": "reference", "unavailable": "oracle/_ref/diamond not present in the snapshot"})
            return
        wl = make_workload(args, 0)
        with tempfile.TemporaryDirectory() as td:
            # thread count: the fastest on a 100 k-query sample (more threads than the CFS quota make the reference slower)
            ns = min(100_000, args.queries)
            qs, d = write_fasta(wl, ns, td)
            cands = sorted({ncpu, min(ncpu, 16), min(ncpu, 32), min(ncpu, 64)})
            tried = {}
            for p in cands:
                tried[p] = min(run_reference(args, qs, d, os.path.join(td, "s.tsv"), p) for _ in range(2 if len(cands) > 1 else 1))
            best_p = min(tried, key=tried.get)
            q, d = write_fasta(wl, args.queries, td)
            warm, steps = min(args.warmup, 1), args.steps
            times = []
            for s in range(warm + steps):
                dt = run_reference(args, q, d, os.path.join(td, "o.tsv"), best_p)
                if s >= warm:
                    times.append(dt)
        cells, note = lookup_cells(args, args.queries, best_p)
        T = sum(times)
        val = (cells * len(times) / T / 1e9) if cells else None
        sample = (f"the full configuration: all {args.queries} queries of rank 0's block x {args.db}-protein DB, one reference process per step (FASTA in, fmt 6 out, "
                  f"whole process wall time), -p {best_p} = fastest of {tried} s on a {ns}-query sample; {len(times)} timed run(s) after {warm} warm-up; {note}")
        emit(({"impl": "reference", "metric": metric, "value": val, "unit": "GCUPS", "n_gpus": args.gpus, "steps": len(times),
                          "warmup": warm, "ms_per_step": 1e3 * T / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "int8/int16 saturating SIMD (AVX2)", "data": "synthetic", "config": dict(config, reference_threads=best_p, sample=sample, same_config=True),
                          "cpu_baseline": {"value": val, "unit": "GCUPS", "cores": best_p, "kind": "reference", "sample": sample},
                          "e2e": {"value": val, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import numpy as np
    import torch
    from diamond_b200 import api

    if args.emit_cells:
        # cell counts of rank 0's block for the given reference thread counts (seedp_bits follows -p), and of the 100 k sample
        wl = make_workload(args, 0)
        tab = load_cells(args.cells_json)
        for p in [int(x) for x in args.emit_cells.split(",")]:
            ctx = api.Context(device=0, threads=p, masking=args.masking, motif_masking=args.masking, **wl["ctx"])
            _, _, st = ctx.blastp(wl["q_raw"], wl["q_lim"], wl["r_raw"], wl["r_lim"])
            ctx.close()
            tab[cells_key(args, args.queries, p)] = st["cells_round1"] + st["cells_round2"]
        if args.cells_json:
            json.dump(tab, open(args.cells_json, "w"), indent=1, sort_keys=True)
        emit(tab)
        return

    torch.cuda.set_device(local)
    from diamond_b200 import shard
    bus = None
    try:  # the CUDA device's own PCI address (torch >= 2.1 exposes it)
        pr = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
    except Exception:
        bus = None
    numa_note = shard.pin_to_gpu_numa_node(local, bus) if world > 1 else "one rank: not pinned"  # before the library starts its host threads
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    os.environ.setdefault("DMND_HOST_THREADS", str(max(1, ncpu // world)))
    wl = make_workload(args, rank)
    q_raw, q_lim, r_raw, r_lim = wl["q_raw"], wl["q_lim"], wl["r_raw"], wl["r_lim"]
    if world > 1:
        # host image for the e2e arm (which uploads and masks the reference inside the timed call): one torch broadcast
        from diamond_b200 import shard
        if rank != 0:
            r_raw, r_lim = np.zeros(0, np.int8), np.zeros(0, np.int64)
        r_raw, r_lim = shard.broadcast_reference(r_raw, r_lim, dist, device=torch.device("cuda", local))
    # pinned host copies for the e2e path
    q_pin = torch.from_numpy(q_raw).pin_memory().numpy()
    r_pin = torch.from_numpy(r_raw).pin_memory().numpy()
    ctx = api.Context(device=local, threads=ref_threads, masking=args.masking, motif_masking=args.masking, **wl["ctx"])

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_ms = []  # host wall time of every step of the last timed() call (each step ends with a device->host read)

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.timing(reset=True)
        t0 = time.perf_counter()
        e0.record()
        last = None
        step_ms.clear()
        for _ in range(n):
            ts = time.perf_counter()
            last = fn()
            step_ms.append(round((time.perf_counter() - ts) * 1e3, 2))
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = max(e0.elapsed_time(e1), 0.0)
        ms = max(ms, 0.0) if ms > 0.5 * wall * 1e3 else wall * 1e3  # events sit on torch's idle stream: fall back to wall if skewed
        if world > 1:
            tt = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt.item())
        return ms, last, ctx.timing()

    # resident blocks.  N > 1: rank 0 loads and masks the reference block, every other rank receives the RESIDENT block -- masked
    # letters, soft table, bias -- device to device over NVLink by the library's own NCCL broadcast (dmnd_block_broadcast): the
    # one collective of the path
    qb = ctx.upload(q_raw, q_lim)
    rb = ctx.upload(r_raw, r_lim) if (world == 1 or rank == 0) else None
    q_res, r_res = q_raw, r_raw
    mask_info = None
    bcast_ms = None
    if args.masking:
        # making the blocks resident includes masking them (what the reference does when it loads a block); the host images
        # the resident call reads (chaining link scores of the host-path queries) are the equally masked letters
        torch.cuda.synchronize()
        t0 = time.perf_counter(); nmq = len(ctx.mask_block(qb, 5, 0, len(q_lim) - 1)); t1 = time.perf_counter()
        nmr = len(ctx.mask_block(rb, 5, 0, len(r_lim) - 1)) if rb is not None else 0
        t2 = time.perf_counter()
        mask_info = {"query_block_ms": round((t1 - t0) * 1e3, 2), "reference_block_ms": round((t2 - t1) * 1e3, 2), "letters_masked": [nmq, nmr],
                     "note": "dmnd_block_mask (tantan + motif table) of the whole block incl. the position list download, one call each, host wall"}
        q_res = ctx.download_letters(qb, q_raw.size)
    if world > 1:
        torch.cuda.synchronize(); dist.barrier()
        t0 = time.perf_counter()
        rb, raw_len, r_lim_b = shard.broadcast_reference_block(ctx, dist, torch.device("cuda", local), rb)
        torch.cuda.synchronize(); dist.barrier()
        bcast_ms = round((time.perf_counter() - t0) * 1e3, 2)
        assert raw_len == r_raw.size and np.array_equal(r_lim_b, r_lim)
    if args.masking:
        r_res = ctx.download_letters(rb, r_raw.size)
    step_res = lambda: ctx.blastp_resident(qb, rb, q_res, q_lim, r_res, r_lim)
    step_e2e = lambda: ctx.blastp(q_pin, q_lim, r_pin, r_lim)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    for _ in range(args.warmup):
        step_res()
    c0 = clocks.mark()
    ms, (m, tr, st), tm = timed(step_res, args.steps)
    step_ms_res = list(step_ms)
    dumped = sample_matches(m, tr) if args.dump_outputs and rank == 0 else None
    c1 = clocks.mark()
    clk = clocks.stop(max(c0 - 1, 0), c1 + 1) if rank == 0 else None
    for _ in range(min(args.warmup, 2)):  # the e2e path has its own first-call allocations (block pool, staging)
        step_e2e()
    ms_e2e, (m2, _, st2), tm2 = timed(step_e2e, args.steps)
    step_ms_e2e = list(step_ms)
    cells = st["cells_round1"] + st["cells_round2"]
    tot = torch.tensor([float(cells), float(st2["cells_round1"] + st2["cells_round2"])], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tot)
    cells_all, cells_all_e2e = float(tot[0].item()), float(tot[1].item())
    value = cells_all * args.steps / (ms / 1e3) / 1e9
    e2e = cells_all_e2e * args.steps / (ms_e2e / 1e3) / 1e9
    # kernel time for the roofline: query lanes overlap on the device, so their stream times cannot be added up; the kernels
    # are timed in a separate pass with ONE lane (every kernel of the step serialised on one stream, same work)
    lanes_env = os.environ.get("DMND_LANES")
    os.environ["DMND_LANES"] = "1"
    # up to three single-lane steps, each timed on its own; the one with the least kernel time is reported (a step is deterministic work:
    # anything above the minimum is a stall of the box -- sporadic 100-300 ms hiccups were seen on this pool -- not kernel time)
    rpasses = max(1, min(args.steps, 3))
    rsteps = 1
    step_res()
    passes = [timed(step_res, 1)[2] for _ in range(rpasses)]
    tm1 = min(passes, key=lambda t: t["dp_score_ms"] + t["dp_trace_ms"] + t["seed_ms"])
    if lanes_env is None:
        del os.environ["DMND_LANES"]
    else:
        os.environ["DMND_LANES"] = lanes_env
    ctx.free_block(qb); ctx.free_block(rb)

    out = None
    if rank == 0:
        # ---- roofline of the dominant kernels (banded SWIPE): integer-ALU bound, see DESIGN.md 4.
        # achieved = lane-ops of the recurrence on the ALGORITHMIC cells of the problems the kernels were LAUNCHED on (a fused query's
        # problem is evaluated once, by the traceback kernel): 9 per score-only cell, 13 per traceback cell (SURVEY 8d), divided by the
        # event-timed DP time of the single-lane pass.  peak = 4 lane-ops x the live-measured issue rate of VIADDMNMX.S16x2 (two 16-bit
        # cells per lane and instruction, two lane-ops each); frac_s32_peak = against 2 x the rate of the 32-bit form (round 1's figure).
        dp_ms = (tm1["dp_score_ms"] + tm1["dp_trace_ms"]) / rsteps
        laneops = (9 * tm1["dp_cells_score"] + 13 * tm1["dp_cells_trace"]) / rsteps
        launched = (tm1["dp_cells_score"] + tm1["dp_cells_trace"]) / rsteps
        peak16, peak32 = 4.0 * ctx.int_peak(packed=True), 2.0 * ctx.int_peak()
        ach = laneops / (dp_ms / 1e3) / 1e12 if dp_ms > 0 else None
        ncu = {}
        try:
            ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic_r2.json")))
        except Exception:
            pass
        roofline = {"bound": "int-alu", "kernel": "swipe16_kernel<R,TRACE> + walk_kernel (banded SWIPE, packed 16-bit DPX lanes; int32 kernels as overflow cascade)",
                    "achieved": ach, "peak": peak16, "unit": "Tlaneop/s", "frac": (ach / peak16) if (ach and peak16) else None,
                    "frac_s32_peak": (ach / peak32) if (ach and peak32) else None, "peak_s32": peak32,
                    "traffic": ncu.get("swipe16_bytes_per_launch"), "traffic_note": ncu.get("note", "no ncu capture committed for this round yet"),
                    "kernel_ms_per_step": dp_ms, "cells_launched_per_step": launched,
                    "padding_factor": (tm1["dp_cells_padded"] / max(1, tm1["dp_cells_score"] + tm1["dp_cells_trace"])),
                    "overflow_reruns": tm1["dp_overflow_reruns"],
                    "kernel_gcups": launched / (dp_ms / 1e3) / 1e9 if dp_ms > 0 else None,
                    "timed": f"CUDA events on the library stream, the fastest of {rpasses} single-lane step(s) after the timed region"}
        # ---- roofline of the seed stage: HBM bound by SURVEY 8d's byte model of the double-indexed join, per shape and block pair:
        # 1 B per letter of both blocks + 36 B per seed entry (write, partition pass, join read) + 96 B of fingerprints per (q, s) pair
        # + 98 B per stage-1 survivor (left-most windows) + 15 B per hit
        sd = st["seed"]
        nshapes = int(ctx.params.n_shapes)
        letters = int(q_raw.size + r_raw.size)
        seed_bytes = nshapes * letters * (1 + 36) + 96 * sd["seed_hits"] + 98 * sd["tentative_matches1"] + 15 * sd["tentative_matches3"]
        seed_ms = tm1["seed_ms"] / rsteps
        try:
            hbm_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 0)) or 6486.0
            hbm_src = "MEASURED_PEAKS.json"
        except Exception:
            hbm_peak, hbm_src = 6486.0, "fallback (B200_PROFILING.md)"
        seed_ach = seed_bytes / (seed_ms / 1e3) / 1e9 if seed_ms > 0 else None
        roofline_seed = {"bound": "hbm", "kernel": "seed stage (ref index build + probe + mask + stage 1/2 + x-drop + hit sort)", "achieved": seed_ach, "peak": hbm_peak,
                         "peak_source": hbm_src, "unit": "GB/s", "frac": (seed_ach / hbm_peak) if seed_ach else None, "algorithmic_bytes_per_step": seed_bytes,
                         "kernel_ms_per_step": seed_ms, "traffic": ncu.get("probe_bytes_per_launch"),
                         "note": "the byte model is the REFERENCE algorithm's (materialised seed arrays); this implementation probes a Bloom filter + bucket directory "
                                 "instead and is bound by issue rate / L2 sector reads (DESIGN.md 4), so frac understates nothing but is far from HBM speed"}
        cpu = None
        if world == 1 and not args.no_cpu_baseline and os.path.exists(REF_BIN):
            n = min(args.sample, args.queries)
            ws = make_workload(args, rank, n)
            sctx = api.Context(device=local, threads=ref_threads, masking=args.masking, motif_masking=args.masking, **ws["ctx"])
            sm, _, sst = sctx.blastp(ws["q_raw"], ws["q_lim"], ws["r_raw"], ws["r_lim"])
            sctx.close()
            scells, tsv = sst["cells_round1"] + sst["cells_round2"], fmt6_of(ws, sm)
            with tempfile.TemporaryDirectory() as td:
                q, d = write_fasta(ws, n, td)
                dt = run_reference(args, q, d, os.path.join(td, "o.tsv"), ref_threads)
                same = open(os.path.join(td, "o.tsv")).read() == tsv
            cpu = {"value": scells / dt / 1e9, "unit": "GCUPS", "cores": ref_threads, "kind": "reference",
                   "sample": f"first {n} queries x full DB, one reference run (FASTA in, fmt 6 out), wall {dt:.2f} s; fmt-6 identical to ours: {same}"}
        # the cell count of this configuration for the reference arm (which must not load the CUDA library)
        if args.cells_json:
            tab = load_cells(args.cells_json)
            tab[cells_key(args, args.queries, ref_threads)] = cells
            json.dump(tab, open(args.cells_json, "w"), indent=1, sort_keys=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumped)
        out = {"metric": metric, "value": value, "unit": "GCUPS", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "int16 (packed DPX lanes, exact: overflow cascades to the int32 kernels; reference int8/int16 lane semantics)",
               "data": "synthetic", "config": config, "clocks": clk,
               "e2e": {"value": e2e, "unit": "GCUPS", "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": tm2["h2d_bytes"] // args.steps,
                       "d2h_bytes_per_step": tm2["d2h_bytes"] // args.steps},
               "gpu_launches": int(tm["launches"]), "roofline": roofline, "roofline_seed": roofline_seed, "cpu_baseline": cpu,
               "step_ms": {"resident": step_ms_res, "e2e": step_ms_e2e}, "masking_ms": mask_info, "reference_broadcast_ms": bcast_ms, "host_pinning_rank0": numa_note,
               "breakdown_ms_per_step": {"seed_stage": st["seed_ms"], "host_bridge": st["host_bridge_ms"], "dp_round1": st["dp1_ms"], "dp_round2": st["dp2_ms"], "total": st["total_ms"]},
               "work": {"cells_per_gpu": cells, "dp_problems_round1": st["dp_problems_round1"], "dp_problems_round2": st["dp_problems_round2"], "dp_problems_fused": st["dp_problems_fused"],
                        "note": "cells = sum band x cols over the reference's round-1 and round-2 problem lists (dp/dp.h:121-124): a property of the workload, "
                                "the same for both arms; fused queries evaluate a surviving problem's matrix once (with traceback) instead of twice",
                        "alignments": int(len(m)), "hits": st["hits"], "seed_counters": {k: int(v) for k, v in st["seed"].items()}, "targets": st["targets"]}}
        emit(out)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
