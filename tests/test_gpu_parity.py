"""Parity of the CUDA path (libcoverm_b200.so through its C ABI / the `coverm` binary) with
 (1) the reference's own golden vectors (tests/golden/reference_cases.py), and
 (2) the CPU oracle on seeded synthetic BAMs (bamgen) that exercise what the tiny fixtures cannot: contigs spanning
     many 8192-element chunks, chunks holding many contigs, deep pile-ups, every filter mode, genome modes.
Outputs are compared as text: identical digit strings mean bit-exact integers AND bit-identical f32 results
(stronger than the 1e-6 relative tolerance BASELINE.json asks for floating-point methods)."""
import os
import subprocess

import pytest

import coverm_b200
from case_runner import DATA, ORACLE_BIN, check_case, run_case
from reference_cases import CASES, CLI_CASES, FILTER_CASES

pytestmark = pytest.mark.gpu

GPU_CASES = [c for c in CASES + CLI_CASES + FILTER_CASES if c["sub"] in ("contig", "genome", "filter-names")]


@pytest.mark.parametrize("case", GPU_CASES, ids=[f"{c['sub']}@{c['ref']}" for c in GPU_CASES])
def test_cuda_path_matches_reference_golden(case):
    check_case(case, run_case(coverm_b200.COVERM_BIN, case, extra_args=["-t", "4"]))


# ---------------------------------------------------------------------------------------------- GPU vs oracle
def _both(argv, threads="8", env=None):
    g = subprocess.run([coverm_b200.COVERM_BIN] + argv + ["-t", threads, "--print-reads-mapped"], capture_output=True,
                       text=True, timeout=900, env=dict(os.environ, **(env or {})))
    o = subprocess.run([ORACLE_BIN] + argv + ["-t", threads, "--print-reads-mapped"], capture_output=True, text=True,
                       timeout=900)
    return g, o


def _assert_same(argv, env=None):
    g, o = _both(argv, env=env)
    assert g.returncode == o.returncode, f"{argv}: exit {g.returncode} vs oracle {o.returncode}\n{g.stderr[-1500:]}"
    if g.stdout != o.stdout:
        gl, ol = g.stdout.splitlines(), o.stdout.splitlines()
        diff = [(i, a, b) for i, (a, b) in enumerate(zip(gl, ol)) if a != b][:8]
        raise AssertionError(f"{argv}: {len(gl)} vs {len(ol)} lines; first differences (line, gpu, oracle): {diff}")
    rm = lambda p: [l for l in p.stderr.splitlines() if l.startswith("#reads_mapped")]
    assert rm(g) == rm(o)
    return g


ALL_METHODS = ["mean", "trimmed_mean", "covered_fraction", "covered_bases", "variance", "length", "count",
               "reads_per_base", "rpkm", "tpm", "anir"]

FIXTURE_RUNS = [
    ["contig", "-m"] + ALL_METHODS + ["-b", DATA + "/1.bam"],
    ["contig", "-m"] + ALL_METHODS + ["-b", DATA + "/eg2.bam", "--output-format", "sparse"],
    ["contig", "-m", "mean", "variance", "-b", DATA + "/1.bam", "--min-read-percent-identity", "95",
     "--min-read-aligned-length", "50"],
    ["contig", "-m", "mean", "trimmed_mean", "-b", DATA + "/eg2.bam", "--proper-pairs-only",
     "--min-read-percent-identity-pair", "0.9", "--min-read-aligned-length-pair", "100"],
    ["contig", "-m", "coverage_histogram", "-b", DATA + "/1read_of_pair_mapped.bam"],
    ["contig", "-m", "metabat", "-b", DATA + "/1.bam", DATA + "/1read_of_pair_mapped.bam"][:5],
    ["genome", "--single-genome", "-m", "mean", "trimmed_mean", "variance", "covered_fraction", "-b", DATA + "/1.bam",
     "--min-covered-fraction", "0"],
    ["contig", "-m", "mean", "trimmed_mean", "--contig-end-exclusion", "0", "--trim-min", "10", "--trim-max", "90",
     "-b", DATA + "/1.bam", "--no-zeros"],
]


@pytest.mark.parametrize("argv", FIXTURE_RUNS, ids=[" ".join(a[:6]).replace(DATA + "/", "") + f"#{i}" for i, a in enumerate(FIXTURE_RUNS)])
def test_cuda_path_matches_oracle_on_reference_fixtures(argv):
    _assert_same(argv)


@pytest.fixture(scope="module")
def synth(tmp_path_factory):
    d = tmp_path_factory.mktemp("synth")
    out = {}

    def gen(name, *args):
        p = str(d / f"{name}.bam")
        subprocess.check_call([coverm_b200.BAMGEN_BIN, "--out", p, "--threads", "8"] + [str(a) for a in args],
                              stdout=subprocess.DEVNULL)
        out[name] = p

    # many small contigs (several per chunk), a few long ones (hundreds of chunks), deep coverage, genomes
    gen("small", "--contigs", 3000, "--reads", 200000, "--seed", 11, "--median-len", 2500, "--min-len", 200, "--max-len", 60000)
    gen("tiny", "--contigs", 4000, "--reads", 60000, "--seed", 12, "--median-len", 300, "--min-len", 90, "--max-len", 2000, "--read-len", 80)
    gen("long", "--contigs", 12, "--reads", 300000, "--seed", 13, "--median-len", 900000, "--sigma", 0.6, "--min-len", 50000, "--max-len", 5000000)
    gen("deep", "--contigs", 40, "--reads", 600000, "--seed", 14, "--median-len", 9000, "--min-len", 2000, "--max-len", 40000)
    gen("mags", "--contigs", 2500, "--genomes", 60, "--reads", 250000, "--seed", 15, "--median-len", 8000, "--definition-out", str(d / "mags.tsv"))
    out["mags_def"] = str(d / "mags.tsv")
    return out


SYNTH_RUNS = [
    ("small", ["contig", "-m"] + ALL_METHODS),
    ("small", ["contig", "-m", "mean", "trimmed_mean", "variance", "--contig-end-exclusion", "0"]),
    ("small", ["contig", "-m", "mean", "trimmed_mean", "covered_fraction", "--min-read-percent-identity", "97", "--min-mapq", "20"]),
    ("small", ["contig", "-m", "mean", "variance", "--proper-pairs-only", "--min-read-aligned-length-pair", "250", "--min-read-percent-identity-pair", "95"]),
    ("small", ["contig", "-m", "mean", "count", "--proper-pairs-only", "--min-mapq", "30", "--min-read-aligned-percent", "95"]),
    ("small", ["contig", "-m", "mean", "trimmed_mean", "--exclude-supplementary", "--include-secondary", "--no-zeros", "--output-format", "sparse"]),
    ("small", ["contig", "-m", "coverage_histogram"]),
    ("small", ["contig", "-m", "metabat"]),
    ("tiny", ["contig", "-m"] + ALL_METHODS),
    ("tiny", ["contig", "-m", "mean", "trimmed_mean", "variance", "--contig-end-exclusion", "10", "--trim-min", "0.2", "--trim-max", "0.8"]),
    ("long", ["contig", "-m"] + ALL_METHODS),
    ("long", ["contig", "-m", "coverage_histogram"]),
    ("deep", ["contig", "-m", "mean", "trimmed_mean", "variance", "covered_fraction"]),
    ("deep", ["contig", "-m", "coverage_histogram", "--min-covered-fraction", "0"]),
    ("mags", ["genome", "-s", "~", "-m", "relative_abundance", "mean", "trimmed_mean", "variance", "covered_fraction", "covered_bases", "length", "count", "rpkm", "tpm", "--min-covered-fraction", "0"]),
    ("mags", ["genome", "-s", "~", "-m", "mean", "trimmed_mean", "--min-read-percent-identity", "95", "--output-format", "sparse", "--no-zeros"]),
    ("mags", ["genome", "--genome-definition", "{mags_def}", "-m", "relative_abundance", "mean", "trimmed_mean", "variance", "--min-covered-fraction", "5"]),
    ("mags", ["genome", "-s", "~", "-m", "coverage_histogram"]),
    ("mags", ["genome", "--single-genome", "-m", "mean", "variance", "trimmed_mean", "--min-covered-fraction", "0"]),
]


@pytest.mark.parametrize("which,argv", SYNTH_RUNS, ids=[f"{w}:{' '.join(a[:7])}#{i}" for i, (w, a) in enumerate(SYNTH_RUNS)])
def test_cuda_path_matches_oracle_on_synthetic_bams(synth, which, argv):
    argv = [a.replace("{mags_def}", synth["mags_def"]) for a in argv]
    _assert_same(argv + ["-b", synth[which]])


# ---------------------------------------------------------------------------------------------- decode paths
# BGZF inputs are decoded on the GPU by default (kd_inflate ... kd_extract); CMB_HOST_DECODE=1 forces the host decoder.
DECODE_FIXTURES = ["2seqs.reads_for_seq1.bam", "7seqs.reads_for_seq1_and_seq2.bam", "1.bam", "eg2.bam", "1read_of_pair_mapped.bam",
                   "k141_2005182.bam", "2seqs.bad_read.1.with_supplementary.bam", "tpm_test.bam"]


def _decode_stats(g):
    lines = [l for l in g.stderr.splitlines() if l.startswith("#device_decode") or l.startswith("#decode_")]
    return lines


@pytest.mark.parametrize("name", DECODE_FIXTURES)
def test_device_inflate_matches_zlib_on_reference_fixtures(name):
    g = _assert_same(["contig", "-m", "mean", "trimmed_mean", "variance", "count", "-b", os.path.join(DATA, name)],
                     env={"CMB_PIPELINE_STATS": "1", "CMB_DECODE_VERIFY": "1"})
    st = _decode_stats(g)
    assert any(l.startswith("#device_decode\tblocks=") for l in st), st  # the device path ran and was not declined
    assert any(l.startswith("#decode_verify\t0 of ") for l in st), st     # every device-inflated block equals zlib's output


@pytest.mark.parametrize("which", ["small", "tiny", "long", "deep", "mags"])
def test_device_inflate_matches_zlib_on_synthetic_bams(synth, which):
    g = _assert_same(["contig", "-m", "mean", "trimmed_mean", "count", "-b", synth[which]],
                     env={"CMB_PIPELINE_STATS": "1", "CMB_DECODE_VERIFY": "1"})
    st = _decode_stats(g)
    # at most the block shared by the header text and the first records may need the library's zlib fallback
    assert any(l.startswith("#device_decode\tblocks=") and ("host_blocks=0" in l or "host_blocks=1\t" in l) for l in st), st
    assert any(l.startswith("#decode_verify\t0 of ") for l in st), st


@pytest.mark.parametrize("which,argv", [SYNTH_RUNS[0], SYNTH_RUNS[2], SYNTH_RUNS[10], SYNTH_RUNS[14]],
                         ids=["small-all", "small-filter", "long-all", "mags-genome"])
def test_host_decode_path_matches_oracle(synth, which, argv):
    argv = [a.replace("{mags_def}", synth["mags_def"]) for a in argv]
    g = _assert_same(argv + ["-b", synth[which]], env={"CMB_HOST_DECODE": "1", "CMB_PIPELINE_STATS": "1"})
    assert any(l.startswith("#pipeline") for l in g.stderr.splitlines())


INFLATE_MODES = [(k, m) for k in ("t1", "g8", "w1") for m in ("persistent", "serial")]


@pytest.mark.parametrize("kernel,mode", INFLATE_MODES, ids=[f"{k}-{m}" for k, m in INFLATE_MODES])
def test_every_inflate_kernel_and_launch_mode_matches_zlib(synth, kernel, mode):
    """The three inflate kernels (thread / eight lanes / warp per block) under the two launch disciplines: one persistent launch
    whose lanes wait for their window's arrival flag (64 KB windows here, so that a small file spans many), and one launch
    ordered behind all the copies (what runs under ncu / compute-sanitizer and for single-window files)."""
    env = {"CMB_PIPELINE_STATS": "1", "CMB_DECODE_VERIFY": "1", "CMB_INFLATE": kernel, "CMB_DECODE_WINDOW_KB": "64",
           "CMB_INFLATE_SERIAL": "1" if mode == "serial" else "0"}
    for which in ("small", "mags"):
        g = _assert_same(["contig", "-m", "mean", "trimmed_mean", "count", "-b", synth[which]], env=env)
        st = _decode_stats(g)
        assert any(l.startswith("#device_decode\tblocks=") and ("host_blocks=0" in l or "host_blocks=1\t" in l) for l in st), st
        assert any(l.startswith("#decode_verify\t0 of ") for l in st), st
        assert not any(l.startswith("#decode_status") and "\t31:" in l for l in st), st  # no window wait expired


def test_declined_blocks_get_a_second_device_pass(synth):
    """Blocks the four-streams-per-warp kernel declines are retried with the one-stream-per-warp kernel (larger tables)
    before the host's zlib is asked; CMB_DECODE_RETRY_TEST marks every 7th block as declined to exercise that path."""
    g = _assert_same(["contig", "-m", "mean", "trimmed_mean", "count", "-b", synth["small"]],
                     env={"CMB_PIPELINE_STATS": "1", "CMB_DECODE_VERIFY": "1", "CMB_DECODE_RETRY_TEST": "1"})
    st = _decode_stats(g)
    assert any(l.startswith("#decode_status") and "\t29:" in l for l in st), st
    assert any(l.startswith("#device_decode\tblocks=") and "host_blocks=0" in l for l in st), st
    assert any(l.startswith("#decode_verify\t0 of ") for l in st), st


def test_device_decode_declines_when_memory_is_short(synth):
    """Not enough device memory for the decode buffers -> the sample is declined before anything is accumulated and the
    host decoder takes over (same table)."""
    g = _assert_same(["contig", "-m", "mean", "trimmed_mean", "count", "-b", synth["small"], synth["tiny"]],
                     env={"CMB_PIPELINE_STATS": "1", "CMB_DECODE_MEM_LIMIT_MB": "8"})
    lines = g.stderr.splitlines()
    assert any(l.startswith("#device_decode\tdeclined") and "not enough device memory" in l for l in lines), lines[-6:]
    assert any(l.startswith("#pipeline") for l in lines)


def test_host_decode_path_matches_reference_goldens():
    for case in GPU_CASES[:12]:
        check_case(case, run_case(coverm_b200.COVERM_BIN, case, extra_args=["-t", "4"], env={"CMB_HOST_DECODE": "1"}))


def test_multiple_samples_reuse_the_arena(synth):
    # second sample runs on the arena that K2 re-zeroed while scanning the first (clean-as-you-go)
    _assert_same(["contig", "-m", "mean", "trimmed_mean", "variance", "--output-format", "sparse", "-b", synth["small"],
                  synth["deep"], synth["small"]])
    _assert_same(["contig", "-m", "mean", "trimmed_mean", "-b", DATA + "/7seqs.reads_for_seq1.bam",
                  DATA + "/7seqs.reads_for_seq1_and_seq2.bam"])


def test_in_memory_bam_through_the_c_abi(synth):
    import numpy as np
    buf = np.fromfile(synth["small"], dtype=np.uint8)
    argv = ["contig", "-m", "mean", "trimmed_mean", "covered_fraction", "-b", synth["small"]]
    sess = coverm_b200.Session(device=0, threads=8)
    r1 = sess.run(argv, memory_inputs={synth["small"]: buf})
    r2 = sess.run(argv)
    sess.close()
    want = subprocess.run([ORACLE_BIN] + argv, capture_output=True, text=True, check=True).stdout
    assert r1.status == 0 and r1.out == want and r2.out == want
    assert r1.samples[0]["k2_launches"] == 1 and r1.samples[0]["k1_launches"] >= 1


def test_smoke_entry():
    import __graft_entry__
    __graft_entry__.smoke()


# ---------------------------------------------------------------------------------------------- pair path on the device
PAIR_RUNS = [
    ("small", ["contig", "-m", "mean", "variance", "count", "--proper-pairs-only", "--min-read-aligned-length-pair", "250", "--min-read-percent-identity-pair", "95"]),
    ("small", ["contig", "-m", "mean", "count", "--proper-pairs-only", "--min-mapq", "30", "--min-read-aligned-percent", "95"]),
    ("small", ["contig", "-m", "mean", "trimmed_mean", "--proper-pairs-only", "--min-read-aligned-percent-pair", "0.9", "--min-read-aligned-length", "100"]),
    ("mags", ["genome", "-s", "~", "-m", "mean", "covered_fraction", "--proper-pairs-only", "--min-read-percent-identity-pair", "97", "--min-covered-fraction", "0"]),
    ("deep", ["contig", "-m", "mean", "variance", "--proper-pairs-only", "--min-read-aligned-length-pair", "280"]),
]


@pytest.mark.parametrize("which,argv", PAIR_RUNS, ids=[f"{w}:{' '.join(a[3:8])}#{i}" for i, (w, a) in enumerate(PAIR_RUNS)])
def test_pair_filter_stays_on_the_device(synth, which, argv):
    """Mate matching of ReferenceSortedBamFilter's pair path (filter.rs:117-233) runs on the GPU (cmb_pairs.cuh): the sample is
    decoded by cmb_submit_bgzf, not by the host pipeline, and the table equals the oracle's; the host's own mate matching
    (CMB_HOST_DECODE=1) must agree too."""
    g = _assert_same(argv + ["-b", synth[which]], env={"CMB_PIPELINE_STATS": "1"})
    assert any(l.startswith("#device_decode\tblocks=") for l in g.stderr.splitlines()), g.stderr[-800:]
    _assert_same(argv + ["-b", synth[which]], env={"CMB_HOST_DECODE": "1"})


FILTER_RS_PAIR_SETTINGS = [  # (fixture, --min-read-aligned-length-pair, --min-read-percent-identity-pair, --min-read-aligned-percent-pair): filter.rs:342-599
    ("7seqs.reads_for_seq1_and_seq2.bam", 90, 0.99, 0.0), ("2seqs.bad_read.1.bam", 250, 0.99, 0.0), ("2seqs.bad_read.1.bam", 300, 0.98, 0.0),
    ("2seqs.bad_read.1.with_extra.bam", 0, 0.98, 0.94), ("2seqs.bad_read.1.bam", 299, 0.98, 0.0), ("eg2.bam", 1, 0.0, 0.0), ("1.bam", 120, 0.95, 0.9),
]


@pytest.mark.parametrize("bam,length,identity,percent", FILTER_RS_PAIR_SETTINGS, ids=[f"{b}:{l}:{i}:{p}" for b, l, i, p in FILTER_RS_PAIR_SETTINGS])
def test_pair_filter_settings_of_the_reference_tests_on_the_device(bam, length, identity, percent):
    """The fixtures and thresholds of the reference's pair-filter unit tests (filter.rs:342-599; the oracle reproduces their
    qname sequences, tests/test_oracle_golden.py) through the device's mate matching: read counts and coverage as the oracle."""
    argv = ["contig", "-m", "mean", "count", "covered_bases", "--proper-pairs-only", "--min-covered-fraction", "0"]
    if length:
        argv += ["--min-read-aligned-length-pair", str(length)]
    if identity:
        argv += ["--min-read-percent-identity-pair", str(identity)]
    if percent:
        argv += ["--min-read-aligned-percent-pair", str(percent)]
    g = _assert_same(argv + ["-b", os.path.join(DATA, bam)], env={"CMB_PIPELINE_STATS": "1"})
    assert any(l.startswith("#device_decode\tblocks=") for l in g.stderr.splitlines()), g.stderr[-800:]


# ---------------------------------------------------------------------------------------------- coverm filter
def _bam_records(path):
    """(header bytes, [record bytes]) of a BAM file, via zlib."""
    import struct
    import zlib
    raw = open(path, "rb").read()
    data, o = bytearray(), 0
    while o < len(raw):
        bsize = struct.unpack_from("<H", raw, o + 16)[0] + 1
        data += zlib.decompress(raw[o + 18:o + bsize - 8], -15)
        o += bsize
    l_text = struct.unpack_from("<I", data, 4)[0]
    n_ref = struct.unpack_from("<I", data, 8 + l_text)[0]
    p = 12 + l_text
    for _ in range(n_ref):
        p += 8 + struct.unpack_from("<I", data, p)[0]
    header, recs = bytes(data[:p]), []
    while p < len(data):
        bs = struct.unpack_from("<I", data, p)[0]
        recs.append(bytes(data[p:p + 4 + bs]))
        p += 4 + bs
    return header, recs


FILTER_RUNS = [
    ("small", ["--min-read-percent-identity", "97", "--min-read-aligned-length", "100"]),
    ("small", ["--min-read-percent-identity", "97", "--inverse"]),
    ("small", ["--proper-pairs-only", "--min-read-aligned-length-pair", "250", "--min-read-percent-identity-pair", "95"]),
    ("small", ["--proper-pairs-only", "--min-read-aligned-length-pair", "280", "--inverse"]),
    ("small", ["--min-mapq", "30"]),
    ("deep", ["--proper-pairs-only", "--min-mapq", "20", "--min-read-aligned-percent", "95", "--exclude-supplementary"]),
    ("mags", []),
]


@pytest.mark.parametrize("which,extra", FILTER_RUNS, ids=[f"{w}:{' '.join(e)}#{i}" for i, (w, e) in enumerate(FILTER_RUNS)])
def test_coverm_filter_on_the_device(synth, tmp_path, which, extra):
    """`coverm filter` (coverm.rs:408-472): the records the device returns, in its order, are exactly the records the oracle's
    ReferenceSortedBamFilter returns (same names in the same order, byte-identical records, the input's header) -- and the
    host's own filter loop (CMB_HOST_DECODE=1) writes the same file content."""
    outs = []
    for env in ({}, {"CMB_HOST_DECODE": "1"}):
        out = str(tmp_path / f"out{len(outs)}.bam")
        p = subprocess.run([coverm_b200.COVERM_BIN, "filter", "-b", synth[which], "-o", out, "-t", "8", "--timing"] + extra, capture_output=True, text=True,
                           timeout=900, env=dict(os.environ, **env))
        assert p.returncode == 0, p.stderr[-800:]
        assert ("device=1" in p.stderr) == (not env), p.stderr[-300:]
        outs.append(_bam_records(out))
    names = subprocess.run([ORACLE_BIN, "filter-names", "-b", synth[which]] + extra, capture_output=True, text=True, timeout=900)
    assert names.returncode == 0, names.stderr[-500:]
    want = names.stdout.split("\n")[:-1]
    in_header, in_recs = _bam_records(synth[which])
    for header, recs in outs:
        assert header == in_header
        got = [r[36:36 + r[12] - 1].decode() for r in recs]
        assert got == want
    assert outs[0][1] == outs[1][1]
    by_bytes = set(in_recs)
    assert all(r in by_bytes for r in outs[0][1][:2000])


def test_histogram_buffer_overflow_grows_and_retries(synth):
    """CMB_TEST_SMALL_HIST starts the device's histogram record / overflow / pair buffers tiny: the first attempt overflows
    (CMB_E_CAPACITY), the library enlarges them (cmb_grow_buffers) and the kernels run again over the tuples still in HBM."""
    for argv in (["contig", "-m", "mean", "trimmed_mean", "variance", "-b", synth["deep"]], ["contig", "-m", "coverage_histogram", "-b", synth["small"]]):
        g = _assert_same(argv, env={"CMB_TEST_SMALL_HIST": "1", "CMB_PIPELINE_STATS": "1"})
        assert "#capacity_retry" in g.stderr, g.stderr[-600:]


def test_arena_beyond_2_pow_32_elements(tmp_path):
    """The north-star reference (906 000 contigs / 5.0 Gbp: the delta arena holds more than 2^32 elements, so every element index of
    K1 / K2 / the TMA row coordinate is exercised beyond 32 bits) with 10 M reads, the whole table against the oracle.  `bench.py
    --config ns` repeats this at 52.6 M reads in every run (`"parity": true`)."""
    import json
    p = str(tmp_path / "ns10m.bam")
    out = subprocess.run([coverm_b200.BAMGEN_BIN, "--out", p, "--threads", "16", "--contigs", "906000", "--reads", "10000000", "--seed", "20260925",
                          "--median-len", "4000", "--sigma", "0.8", "--min-len", "1000", "--max-len", "2000000"],
                         check=True, capture_output=True, text=True).stdout
    info = json.loads(out.strip().splitlines()[-1])
    assert info["bases"] > 2 ** 32 and info["records"] >= 10_000_000, info
    try:
        g, o = _both(["contig", "-m", "mean", "trimmed_mean", "covered_fraction", "variance", "-b", p], threads="16",
                     env={"CMB_PIPELINE_STATS": "1"})
        assert g.returncode == o.returncode == 0, g.stderr[-1500:]
        assert g.stdout == o.stdout
        assert any(l.startswith("#device_decode\tblocks=") for l in g.stderr.splitlines())  # decoded on the device, not declined
    finally:
        os.remove(p)
