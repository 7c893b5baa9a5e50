"""The drop-in command line (ngsdist_b200/bin/ngsDist): same flags, inputs and .dist layout as the reference.

CPU part: argument validation reproduces parse_args.cpp:203-220 (message + exit status 255) before any CUDA call.
GPU part: every golden case is run through the binary and compared with the reference's own .dist text; inputs made up
inside a test are compared with the .dist text the reference writes for them, as the CPU oracle restates it.
"""
import gzip
import os
import subprocess

import numpy as np
import pytest

import oracle
from util import GOLDEN, format_dist, golden_text, manifest, parse_flags

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "ngsdist_b200", "bin", "ngsDist")
MAN = manifest()


def run_cli(args, **kw):
    return subprocess.run([CLI] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, **kw)


def reference_text(data, flags, labels=None, **kw):
    """The reference's .dist text for `data` run with the compute `flags`: the CPU oracle through the reference's writer,
    which reproduces every .dist in tests/golden/ (written by the unmodified reference) byte for byte
    (tests/test_oracle_golden.py).  kw: kind=1 for text input, genotypes=True for {-1,0,1,2} codes."""
    okw, _ = parse_flags(flags)
    return format_dist([r["dist"] for r in oracle.run_job(data, **okw, **kw)], labels)


def test_cli_is_built():
    assert os.path.exists(CLI), "run __graft_entry__.build()"


@pytest.mark.parametrize("args,msg", [
    ([], "genotype input file (--geno) missing!"),
    (["--geno", "x.bin"], "number of individuals (--n_ind) missing!"),
    (["--geno", "x.bin", "--n_ind", "3"], "number of sites (--n_sites) missing!"),
    (["--geno", "x.bin", "--n_ind", "3", "--n_sites", "4", "--tot_sites", "9", "--pairwise_del", "--out", "o"], "cannot specify total number of sites"),
    (["--geno", "x.gz", "--n_ind", "3", "--n_sites", "4", "--call_geno", "--out", "o"], "can only call genotypes from likelihoods/probabilities!"),
    (["--geno", "x.bin", "--n_ind", "3", "--n_sites", "4", "--evol_model", "9", "--out", "o"], "invalid correction method specified!"),
    (["--geno", "x.bin", "--n_ind", "3", "--n_sites", "4", "--evol_model", "3", "--out", "o"], "requires position information!"),
    (["--geno", "x.bin", "--n_ind", "3", "--n_sites", "4"], "output prefix (--out) missing!"),
    (["--geno", "x.bin", "--n_ind", "3", "--n_sites", "4", "--out", "o", "--n_threads", "0"], "number of threads cannot be less than 1!"),
    # single-dash long options and unique prefixes are accepted (getopt_long_only), then the size check fires
    (["-geno", os.path.join(GOLDEN, "g7x53.bin"), "-n_ind", "7", "-n_sites", "50", "-out", "o", "-verb", "0"], "invalid/corrupt genotype input file!"),
])
def test_cli_argument_errors(args, msg):
    r = run_cli(args + ([] if "-verb" in args else ["--verbose", "0"]))
    assert r.returncode == 255
    assert "ERROR: [" in r.stderr and msg in r.stderr


def test_cli_io_selftest_exact_formatter_and_parser():
    """The writer's exact fast "%.10f" and the reader's fast number parser against libc on 2e6 random values (+ specials,
    decimal half-way points, non-numbers): must be byte / bit identical (SURVEY §8f N1, N2)."""
    r = run_cli(["--selftest_io", "2000000"])
    assert r.returncode == 0, r.stderr[-2000:]
    assert "0 mismatches" in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in MAN["binary"] + MAN["text"] if c["n_sites"] > 64][:6], ids=lambda c: c["name"])
def test_cli_chunked_threaded_reader(case, tmp_path):
    """Many 64-site chunks through the double-buffered reader thread (NGSD_CLI_CHUNK) give the same file as one chunk."""
    outs = []
    for chunk in ("64", "1000000"):
        out = str(tmp_path / ("out%s.dist" % chunk))
        args = ["--geno", os.path.join(GOLDEN, case["input"]), "--n_ind", str(case["n_ind"]), "--n_sites", str(case["n_sites"]),
                "--out", out, "--n_threads", "3", "--verbose", "0"] + case["flags"]
        r = run_cli(args, env=dict(os.environ, NGSD_CLI_CHUNK=chunk))
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append(open(out).read())
    assert outs[0] == outs[1]


@pytest.mark.gpu
def test_cli_text_reader_many_chunks_matches_binary_input(tmp_path):
    """C1-style text input (header + 3 leading label columns, gz) read in 64-site chunks by the threaded parser gives
    the same .dist as the same values read from the binary file."""
    import gzip
    from util import load_bin
    n_ind, n_sites = 24, 400
    raw = load_bin("g24x400.bin", n_ind, n_sites)
    txt = str(tmp_path / "g.txt.gz")
    with gzip.open(txt, "wt") as fh:
        fh.write("marker\tallele1\tallele2\t" + "\t".join("Ind%d" % (i // 3) for i in range(n_ind * 3)) + "\n")
        for s in range(n_sites):
            fh.write("chr1_%d\tA\tC\t" % s + "\t".join(repr(float(v)) for v in raw[s].reshape(-1)) + "\n")
    outs = []
    for geno, chunk in ((os.path.join(GOLDEN, "g24x400.bin"), "1000000"), (txt, "64")):
        out = str(tmp_path / ("o%s.dist" % chunk))
        r = run_cli(["--geno", geno, "--probs", "--n_ind", str(n_ind), "--n_sites", str(n_sites), "--out", out, "--n_threads", "4",
                     "--verbose", "0", "--indep_geno", "--n_boot_rep", "2", "--boot_block_size", "10", "--seed", "5"],
                    env=dict(os.environ, NGSD_CLI_CHUNK=chunk))
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append(open(out).read())
    assert outs[0] == outs[1]


@pytest.mark.gpu
@pytest.mark.parametrize("case", MAN["binary"] + MAN["text"], ids=lambda c: c["name"])
def test_cli_reproduces_reference_dist_files(case, tmp_path):
    out = str(tmp_path / "out.dist")
    args = ["--geno", os.path.join(GOLDEN, case["input"]), "--n_ind", str(case["n_ind"]), "--n_sites", str(case["n_sites"]),
            "--out", out, "--n_threads", "4", "--verbose", "0"] + case["flags"]
    r = run_cli(args)
    assert r.returncode == 0, r.stderr[-2000:]
    got_text = open(out).read()
    want_text = golden_text(case["name"])
    got = [m for _, m in oracle.parse_dist(out, case["n_ind"])]
    ref_path = str(tmp_path / "ref.dist")
    open(ref_path, "w").write(want_text)
    want = [m for _, m in oracle.parse_dist(ref_path, case["n_ind"])]
    assert len(got) == len(want)
    # identical layout: same lines, labels, column counts
    assert [l.split("\t")[0] for l in got_text.split("\n")] == [l.split("\t")[0] for l in want_text.split("\n")]
    for g, w in zip(got, want):
        fin = np.isfinite(w)
        assert np.array_equal(np.isnan(g), np.isnan(w)) and np.array_equal(np.isinf(g), np.isinf(w))
        assert np.abs(g[fin] - w[fin]).max() <= 1.1e-10      # at most one unit in the 10th printed decimal
    # The written file is the reference's byte for byte: the CLI redoes the tail of gen_dist (ngsDist.cpp:372-386) with the
    # host's libm on the raw distance, and the device sums agree with the reference's sequential sums far below the 10th
    # printed decimal (a value within ~1e-14 of a "%.10f" rounding boundary could still differ; none of the goldens has one).
    assert got_text == want_text


@pytest.mark.gpu
def test_cli_labels_stdin_and_nan_spelling(tmp_path):
    n_ind, n_sites = 5, 64
    raw = oracle.synth_raw(3, 0.0, n_ind, n_sites)
    raw[:32, 0, :] = 1 / 3
    raw[32:, 1, :] = 1 / 3                      # individuals 0 and 1 never share a site -> cnt == 0 -> -nan / nan
    geno = tmp_path / "in.bin"
    raw.tofile(geno)
    labels = tmp_path / "labels.txt"
    labels.write_text("# comment\nheader\nA\tx\nB\nC\nD\nE\n")
    out = tmp_path / "o.dist"
    flags = ["--probs", "--indep_geno", "--pairwise_del", "--evol_model", "0"]
    r = run_cli(["--geno", str(geno), "--n_ind", "5", "--n_sites", "64", "--labelsH", str(labels), "--out", str(out), "--verbose", "0"] + flags)
    assert r.returncode == 0, r.stderr
    ref_text = reference_text(raw, flags, labels=list("ABCDE"))
    text = out.read_text()
    assert text.split("\n")[2].startswith("A\t0.0000000000\t-nan\t")
    assert [l.split("\t")[0] for l in text.split("\n")] == [l.split("\t")[0] for l in ref_text.split("\n")]
    assert text.count("nan") == ref_text.count("nan") and text.count("-nan") == ref_text.count("-nan")
    # binary from stdin ("-")
    out2 = tmp_path / "o2.dist"
    with open(geno, "rb") as fh:
        r = subprocess.run([CLI, "--geno", "-", "--probs", "--n_ind", "5", "--n_sites", "64", "--labelsH", str(labels), "--out", str(out2),
                            "--verbose", "0"] + flags[1:], stdin=fh, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr
    assert out2.read_text() == text


@pytest.mark.gpu
def test_cli_c1_reference_test_script_matrix(tmp_path):
    """BASELINE configs[0] (C1): the 18 runs of the reference's own examples/test.sh (genotype text, BEAGLE-style text with
    header + 3 leading columns + --pos, binary, plain text posteriors; bootstrap, block size, --call_geno, thresholds) at
    its shape, 24 individuals x 10 000 sites with --labels, on synthetic data (the script's inputs are not shipped, SURVEY
    D4).  Every run is executed by the drop-in CLI and its .dist file is compared with the reference's (reference_text):
    same layout and labels, values within 1e-9 (default --probs rows run the per pair-site EM in both)."""
    import gzip
    n_ind, n_sites = 24, 10000
    raw = oracle.synth_raw(20251018, 0.05, n_ind, n_sites)
    P = raw / raw.sum(axis=2, keepdims=True)
    # keep 6-decimal text values off the --call_thresh 0.9 knife edge (a 1-ulp log/exp difference could flip a call there,
    # SURVEY App. E-7): no triple whose printed maximum is exactly 0.900000
    P[np.round(P, 6).max(axis=2) == 0.9] = (0.91, 0.05, 0.04)
    P6 = np.array(["%.6f" % v for v in P.reshape(-1)]).astype(np.float64).reshape(P.shape)    # the values the text files hold
    label_names = ["ind%02d_pop%d" % (i, i // 8) for i in range(n_ind)]
    labels = str(tmp_path / "testA.labels")
    open(labels, "w").write("".join(l + "\n" for l in label_names))
    # genotype text: chr, position, then one code per individual (-1 = missing where the synthetic triple is uniform)
    geno = np.argmax(raw, axis=2).astype(int)
    geno[(raw[..., 0] == raw[..., 1]) & (raw[..., 1] == raw[..., 2])] = -1
    f_geno = str(tmp_path / "testA_T.geno.gz")
    with gzip.open(f_geno, "wt") as fh:
        for s in range(n_sites):
            fh.write("chrSIM\t%d\t" % (s + 1) + "\t".join(str(g) for g in geno[s]) + "\n")
    f_beagle = str(tmp_path / "testA_2.beagle.gz")
    with gzip.open(f_beagle, "wt") as fh:
        fh.write("marker\tallele1\tallele2\t" + "\t".join("Ind%d" % (i // 3) for i in range(3 * n_ind)) + "\n")
        for s in range(n_sites):
            fh.write("chrSIM_%d\t0\t1\t" % (s + 1) + "\t".join("%.6f" % v for v in P[s].reshape(-1)) + "\n")
    f_pos = str(tmp_path / "testA.pos")
    open(f_pos, "w").write("".join("chrSIM\t%d\n" % (s + 1) for s in range(n_sites)))
    f_bin = str(tmp_path / "testA_32.geno")
    P.tofile(f_bin)
    f_txt = str(tmp_path / "testA_8.geno.gz")
    with gzip.open(f_txt, "wt") as fh:
        for s in range(n_sites):
            fh.write("chrSIM\t%d\t" % (s + 1) + "\t".join("%.6f" % v for v in P[s].reshape(-1)) + "\n")
    boot = [[], ["--n_boot_rep", "5"], ["--n_boot_rep", "5", "--boot_block_size", "10"]]
    call = [["--n_boot_rep", "5", "--boot_block_size", "10", "--call_geno"],
            ["--n_boot_rep", "5", "--boot_block_size", "10", "--call_geno", "--N_thresh", "0.3", "--call_thresh", "0.9"]]
    # name, file, CLI flags, the file's values and how the reference reads them
    runs = [("T%d" % k, f_geno, b, geno, dict(genotypes=True)) for k, b in enumerate(boot)]
    runs += [("2_%d" % k, f_beagle, ["--probs", "--pos", f_pos] + b, P6, dict(kind=1)) for k, b in enumerate(boot + call)]
    runs += [("32_%d" % k, f_bin, ["--probs"] + b, P, dict(kind=0)) for k, b in enumerate(boot + call)]
    runs += [("8_%d" % k, f_txt, ["--probs"] + b, P6, dict(kind=1)) for k, b in enumerate(boot + call)]
    assert len(runs) == 18
    threads = str(os.cpu_count() or 4)
    worst = 0.0
    for name, path, extra, data, read in runs:
        outs = [str(tmp_path / ("%s_b200.dist" % name)), str(tmp_path / ("%s_ref.dist" % name))]
        cmd = [CLI, "--n_threads", threads, "--seed", "12345", "--verbose", "0", "--geno", path, "--n_ind", str(n_ind),
               "--n_sites", str(n_sites), "--labels", labels] + extra + ["--out", outs[0]]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert r.returncode == 0, (name, r.stderr[-1500:])
        compute = [f for f in extra if f not in ("--pos", f_pos)] + ["--seed", "12345"]
        open(outs[1], "w").write(reference_text(data, compute, labels=label_names, **read))
        ta, tb = open(outs[0]).read(), open(outs[1]).read()
        la, lb = ta.split("\n"), tb.split("\n")
        assert len(la) == len(lb), name
        assert [x.split("\t")[0] for x in la] == [x.split("\t")[0] for x in lb], "%s: layout / labels differ" % name
        ma = [m for _, m in oracle.parse_dist(outs[0], n_ind)]
        mb = [m for _, m in oracle.parse_dist(outs[1], n_ind)]
        assert len(ma) == len(mb) == (1 + (5 if "--n_boot_rep" in extra else 0))
        for x, y in zip(ma, mb):
            assert np.array_equal(np.isnan(x), np.isnan(y))
            d = np.nanmax(np.abs(x - y))
            worst = max(worst, float(d))
            assert d <= 1e-9 * max(1.0, float(np.nanmax(np.abs(y)))) + 1.01e-10, (name, d)   # + one unit of the 10th printed decimal
    print("C1 test.sh matrix: 18 runs, worst |difference| of printed values %.3g" % worst)


@pytest.mark.gpu
def test_cli_plink_bed_input_matches_genotype_text(tmp_path):
    """Extension (SURVEY §8f N3): a variant-major PLINK .bed (2-bit genotypes) gives byte for byte the .dist of the same
    genotypes as {-1,0,1,2} text -- which the reference binary reads too, so the chain bed -> text -> reference is pinned."""
    import gzip
    from ngsdist_b200 import pack_genotypes
    rng = np.random.RandomState(8)
    n_ind, n_sites = 23, 300
    geno = rng.randint(-1, 3, size=(n_sites, n_ind)).astype(np.int8)
    txt = str(tmp_path / "g.geno.gz")
    with gzip.open(txt, "wt") as fh:
        for s in range(n_sites):
            fh.write("\t".join(str(g) for g in geno[s]) + "\n")
    bed = str(tmp_path / "g.bed")
    with open(bed, "wb") as fh:
        fh.write(bytes([0x6c, 0x1b, 0x01]))
        fh.write(pack_genotypes(geno, field_of_code=[1, 0, 2, 3]).tobytes())   # -1 -> 01, 0 -> 00, 1 -> 10, 2 -> 11
    flags = ["--n_ind", str(n_ind), "--n_sites", str(n_sites), "--verbose", "0", "--pairwise_del", "--evol_model", "0",
             "--n_boot_rep", "3", "--boot_block_size", "20", "--seed", "4"]
    texts = []
    for path, env in ((txt, None), (bed, None), (bed, dict(os.environ, NGSD_CLI_CHUNK="64"))):
        out = str(tmp_path / ("o%d.dist" % len(texts)))
        r = run_cli(["--geno", path, "--out", out] + flags, env=env)
        assert r.returncode == 0, r.stderr
        texts.append(open(out).read())
    assert texts[0] == texts[1] == texts[2]
    assert texts[0] == reference_text(geno, flags[6:], genotypes=True)
    # a truncated file and sample-major files are refused
    bad = str(tmp_path / "bad.bed")
    with open(bad, "wb") as fh:
        fh.write(bytes([0x6c, 0x1b, 0x00]))
        fh.write(pack_genotypes(geno, field_of_code=[1, 0, 2, 3]).tobytes())
    r = run_cli(["--geno", bad, "--out", str(tmp_path / "x")] + flags)
    assert r.returncode != 0 and "variant-major" in r.stderr
    r = run_cli(["--geno", bed, "--out", str(tmp_path / "x"), "--n_ind", str(n_ind), "--n_sites", str(n_sites + 1), "--verbose", "0"])
    assert r.returncode != 0 and "invalid/corrupt genotype input file!" in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["GL", "PL"])
@pytest.mark.parametrize("flags", [["--indep_geno", "--pairwise_del"], [], ["--call_geno"]], ids=["indep_pdel", "em", "call"])
def test_cli_vcf_likelihoods_are_the_log_scale_text_input(fmt, flags, tmp_path):
    """Extension (SURVEY §8f N3): FORMAT/GL (log10) or FORMAT/PL (phred) of a VCF enter the front end as natural-log
    likelihoods -- byte-identical output to the same numbers written as a .gz text file and read with --probs --log_scale
    (the reference's own text path, read_data.cpp:83-87,98)."""
    import math
    n_ind, n_sites = 9, 70
    raw = oracle.synth_raw(41, 0.1, n_ind, n_sites)
    rng = np.random.RandomState(1)
    vcf = tmp_path / "in.vcf.gz"
    txt = tmp_path / "in.txt.gz"
    lik = []
    with gzip.open(vcf, "wt") as fv, gzip.open(txt, "wt") as ft:
        fv.write("##fileformat=VCFv4.2\n##FORMAT=<ID=GT,Number=1,Type=String,Description=\"g\">\n")
        fv.write("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join("S%d" % i for i in range(n_ind)) + "\n")
        for s in range(n_sites):
            cols, vals = [], []
            for i in range(n_ind):
                if rng.rand() < 0.1:
                    cols.append("./.:.:3")
                    vals += [repr(math.log(1.0 / 3))] * 3
                    continue
                if fmt == "GL":
                    f = ["%.4f" % math.log10(max(x, 1e-30)) for x in raw[s, i]]
                    L = [float(t) * 2.302585092994046 for t in f]
                else:
                    f = ["%d" % min(255, int(round(-10 * math.log10(max(x, 1e-30))))) for x in raw[s, i]]
                    L = [-float(t) / 10 * 2.302585092994046 for t in f]
                cols.append("0/1:" + ",".join(f) + ":7")
                vals += [repr(v) for v in L]
            fv.write("chr1\t%d\t.\tA\tC\t.\tPASS\t.\tGT:%s:DP\t" % (s + 1, fmt) + "\t".join(cols) + "\n")
            ft.write("\t".join(vals) + "\n")
            lik.append([float(v) for v in vals])
    outs = []
    for path, extra in ((vcf, []), (txt, ["--probs", "--log_scale"])):
        out = str(tmp_path / (os.path.basename(str(path)) + ".dist"))
        r = run_cli(["--geno", str(path), "--n_ind", str(n_ind), "--n_sites", str(n_sites), "--out", out, "--n_threads", "3", "--verbose", "0",
                     "--n_boot_rep", "2", "--boot_block_size", "7", "--seed", "12345"] + extra + flags)
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append(open(out).read())
    assert outs[0] == outs[1]
    # ... and what the reference writes for that text file: the same bytes
    assert outs[0] == reference_text(np.array(lik).reshape(n_sites, n_ind, 3),
                                     ["--probs", "--log_scale", "--n_boot_rep", "2", "--boot_block_size", "7", "--seed", "12345"] + flags, kind=1)


@pytest.mark.gpu
def test_cli_packs_six_decimal_text_posteriors(tmp_path):
    """6-decimal .gz posteriors travel as 3 x 20 bits (NGSD_XFER_U20X3); NGSD_CLI_NO_PACK=1 sends the doubles: same bytes out."""
    case = [c for c in MAN["text"] if c["name"] == "txt_grid_pdel"][0]
    outs = []
    for env in ({}, {"NGSD_CLI_NO_PACK": "1"}):
        out = str(tmp_path / ("o%d.dist" % len(outs)))
        r = subprocess.run([CLI, "--geno", os.path.join(GOLDEN, case["input"]), "--n_ind", str(case["n_ind"]), "--n_sites", str(case["n_sites"]),
                            "--out", out, "--verbose", "0"] + case["flags"], env=dict(os.environ, **env), stdout=subprocess.PIPE,
                           stderr=subprocess.PIPE, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append(open(out).read())
    assert outs[0] == outs[1] == golden_text(case["name"])


@pytest.mark.gpu
def test_cli_tree_flag_writes_one_newick_per_matrix(tmp_path):
    from oracle import nj_oracle
    case = [c for c in MAN["binary"] if c["name"] == "c1_indep_boot"][0]
    out, tree = str(tmp_path / "o.dist"), str(tmp_path / "o.nwk")
    r = run_cli(["--geno", os.path.join(GOLDEN, case["input"]), "--n_ind", str(case["n_ind"]), "--n_sites", str(case["n_sites"]), "--out", out,
                 "--tree", tree, "--verbose", "0"] + case["flags"])
    assert r.returncode == 0, r.stderr[-2000:]
    assert open(out).read() == golden_text(case["name"])
    trees = open(tree).read().strip().split("\n")
    mats = [m for _, m in oracle.parse_dist(out, case["n_ind"])]
    assert len(trees) == len(mats) == 6
    for t, m in zip(trees, mats):                       # the matrices as written (10 decimals) -> the same topology from the CPU restatement
        want = nj_oracle.nj(m)[0]
        assert nj_oracle.newick_lengths(t)[0] == nj_oracle.newick_lengths(want)[0]
        assert np.allclose(nj_oracle.newick_lengths(t)[1], nj_oracle.newick_lengths(want)[1], atol=1e-8)
    # FILE.support: the main tree with the percentage of the 5 bootstrap trees holding each internal edge (README.md:83-98,
    # the raxmlHPC -f b step); the host code behind it is checked against the definition in tests/test_tree_support.py
    import ngsdist_b200 as nb
    assert open(tree + ".support").read() == nb.tree_support(trees[0], trees[1:], percent=True) + "\n"
