import os, subprocess, sys
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
ORACLE_LIB = os.path.join(ROOT, "oracle", "_build", "libdmnd_oracle.so")
PRODUCT_LIB = os.path.join(ROOT, "diamond_b200", "libdmnd_b200.so")
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "diamond")  # the unmodified reference (make ref): only needed to record reference_outputs.json


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle_lib():
    """The TEST-ONLY library: host pipeline linked over the CPU restatement of the kernels (oracle/dmnd_oracle.c)."""
    subprocess.run(["make", "-s", "oracle"], cwd=ROOT, check=True)
    from diamond_b200 import api
    return api.load(ORACLE_LIB)


@pytest.fixture(scope="session")
def product_lib():
    from diamond_b200 import api
    if not os.path.exists(PRODUCT_LIB):
        subprocess.run(["make", "-s", "lib"], cwd=ROOT, check=True)
    return api.load(PRODUCT_LIB)


REFERENCE_OUTPUTS = os.path.join(GOLDEN, "reference_outputs.json")


def text_digest(data, log_text=None, log_patterns=()):
    """{sha256, bytes, lines} of an output file's contents (str or bytes), plus the first group of each --log pattern."""
    import hashlib, re
    b = data.encode() if isinstance(data, str) else data
    d = {"sha256": hashlib.sha256(b).hexdigest(), "bytes": len(b), "lines": b.count(b"\n")}
    if log_patterns:
        d["log"] = [re.search(p, log_text).group(1) for p in log_patterns]
    return d


def reference_output(name, args, log_patterns=(), drop_prefix=None):
    """The digest (text_digest) of what the unmodified reference writes for the command line `args` (without the program and
    `-o`; lines that start with `drop_prefix` left out), as stored in tests/golden/reference_outputs.json together with the
    command line it was recorded with (files by name only: they live in temporary directories).  A test whose command line no
    longer matches its recording fails and says so.  With DMND_RECORD_REFERENCE=1 and the reference built (`make ref`:
    oracle/_ref/diamond), the reference is run on `args` and the stored entry replaced."""
    import json, tempfile
    tab = json.load(open(REFERENCE_OUTPUTS)) if os.path.exists(REFERENCE_OUTPUTS) else {}
    argv = [os.path.basename(a) if os.path.isabs(a) else a for a in args]
    if os.environ.get("DMND_RECORD_REFERENCE") == "1":
        assert os.path.exists(REF_BIN), "DMND_RECORD_REFERENCE=1 needs oracle/_ref/diamond (make ref)"
        with tempfile.TemporaryDirectory() as td:
            out = os.path.join(td, "out")
            r = subprocess.run([REF_BIN] + list(args) + ["-o", out], capture_output=True, text=True, check=True)
            data = open(out, "rb").read()
            if drop_prefix:
                data = b"".join(l for l in data.splitlines(keepends=True) if not l.startswith(drop_prefix.encode()))
            tab[name] = dict(text_digest(data, r.stdout + r.stderr, log_patterns), args=argv)
        with open(REFERENCE_OUTPUTS, "w") as f:
            json.dump(tab, f, indent=1, sort_keys=True)
            f.write("\n")
    assert name in tab, f"no stored reference output {name!r}: record it with DMND_RECORD_REFERENCE=1"
    want = dict(tab[name])
    recorded = want.pop("args")
    assert recorded == argv, f"reference output {name!r} was recorded for {recorded}, the test now runs {argv}: record it again with DMND_RECORD_REFERENCE=1"
    return want


_cache = {}


def workload_blocks(name):
    """(w, q_raw, q_limits, r_raw, r_limits) of a named synthetic workload, cached per session."""
    if name not in _cache:
        from diamond_b200 import api, synth
        w = synth.named(name)
        q_raw, q_lim = api.block_image(w["q_letters"], w["q_off"])
        r_raw, r_lim = api.block_image(w["db_letters"], w["db_off"])
        _cache[name] = (w, q_raw, q_lim, r_raw, r_lim)
    return _cache[name]
