"""The C++ `coverage` command (rows N1-N4): real BAM + FASTA files in, callable_regions.bed + summary.json + summary.html +
SVG plots out, compared with the oracle run on the same records."""
import json
import os
import subprocess

import numpy as np
import pytest

from decodingustools_b200 import synth
from decodingustools_b200.options import CallableOptions
from tests import bamio
from tests.helpers import run_oracle
from tests.test_oracle_vs_naive import random_reads

pytestmark = pytest.mark.gpu
CLI = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "decodingustools_b200", "decodingus-tools-b200")


def _run(tmp_path, contigs, extra_args=(), fasta_contigs=None, index=False):
    """contigs: (name, tid, length, ref, reads)."""
    bam = str(tmp_path / "in.bam"); fa = str(tmp_path / "ref.fa")
    if os.path.exists(bam + ".bai"):
        os.remove(bam + ".bai")
    bamio.write_bam(bam, [(n, l, r) for n, _, l, _, r in contigs], index=index, block=4096 if index else 0xFF00)
    bamio.write_fasta(fa, fasta_contigs if fasta_contigs is not None else [(n, ref) for n, _, _, ref, _ in contigs])
    p = subprocess.run([CLI, "coverage", bam, "-r", fa, "-o", str(tmp_path / "out.bed"), *extra_args], cwd=tmp_path,
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    return open(tmp_path / "out.bed", "rb").read(), json.load(open(tmp_path / "summary.json")), open(tmp_path / "summary.json").read()


def _check(contigs, opt, bed, js):
    o = run_oracle(contigs, opt)
    assert bed == o.bed()
    order, fl, sm = o.export()
    ex = js["export"]
    assert [c["name"] for c in ex["contigs"]] == [o.contigs[i].name for i in order]
    for c, f, i in zip(ex["contigs"], fl, order):
        oc = o.contigs[i]
        assert c["length"] == oc.length and c["unique_reads"] == oc.n_reads and c["covered_bases"] == oc.n_covered_bases
        assert [c["state_distribution"][k] for k in ("ref_n", "callable", "no_coverage", "low_coverage", "excessive_coverage",
                                                     "poor_mapping_quality")] == oc.counts
        assert c["coverage_percent"] == f["coverage_percent"] and c["average_depth"] == f["average_depth"]
        assert c["quality_stats"] == {k: f[k] for k in ("average_mapq", "average_baseq", "q30_percentage")}
    s = ex["summary"]
    assert s["total_bases"] == sm["total_bases"] and s["callable_bases"] == sm["callable_bases"]
    assert s["callable_percentage"] == sm["callable_percentage"] and s["average_depth"] == sm["average_depth"]
    assert s["contigs_analyzed"] == sm["contigs_analyzed"]
    assert ex["quality_metrics"] == {k: sm[k] for k in ("average_mapq", "average_baseq", "q30_percentage")}
    assert ex["total_unique_reads"] == sm["total_unique_reads"]


def test_cli_matches_oracle_on_a_small_genome(tmp_path):
    cs = [synth.synth_short("chr1", 120_000, seed=41), synth.synth_short("chr2", 60_000, seed=42),
          synth.synth_short("chrM", 16_569, seed=43, depth=300.0)]
    contigs = [(c.name, tid, c.length, c.ref, c.reads) for tid, c in enumerate(cs)]
    bed, js, raw = _run(tmp_path, contigs)
    _check(contigs, CallableOptions(), bed, js)
    assert js["export"]["summary"]["aligner"] == "BWA" and js["export"]["summary"]["read_length"] == 150
    assert js["files"]["bed_file"].endswith("out.bed") and '"coverage_percent": ' in raw
    # -L keeps tid order and the largest-contig rule only sees the selected contigs
    sel = [contigs[1], contigs[2]]
    bed, js, raw = _run(tmp_path, contigs, ["-L", "chrM", "-L", "chr2"])
    _check(sel, CallableOptions(), bed, js)
    # with a .bai next to the BAM the reader jumps to the selected contigs: same files
    bed_i, js_i, raw_i = _run(tmp_path, contigs, ["-L", "chrM", "-L", "chr2"], index=True)
    assert bed_i == bed and raw_i == raw


def test_cli_flags_weird_cigars_and_short_reference(tmp_path):
    rng = np.random.default_rng(7)
    length = 3000
    ref = bytes(rng.choice(list(b"ACGTN"), size=length, p=[.24, .24, .24, .24, .04]).tolist())
    reads = random_reads(rng, length, 800, max_len=60)
    contigs = [("chrT", 0, length, ref, reads)]
    opt = CallableOptions(min_depth=2, max_depth=7, min_mapping_quality=5, min_base_quality=12, min_depth_for_low_mapq=4,
                          max_low_mapq=2, max_low_mapq_fraction=0.25)
    args = ["--min-depth", "2", "--max-depth", "7", "--min-mapping-quality", "5", "--min-base-quality", "12",
            "--min-depth-for-low-mapq", "4", "--max-low-mapq", "2", "--max-low-mapq-fraction", "0.25"]
    # the FASTA holds only the first 2000 bases: the rest reads as 'N' (mod.rs:79-80)
    bed, js, _ = _run(tmp_path, contigs, args, fasta_contigs=[("chrT", ref[:2000])])
    _check([("chrT", 0, length, ref[:2000], reads)], opt, bed, js)


def test_cli_errors_like_the_reference(tmp_path):
    c = synth.synth_short("chr1", 20_000, seed=44)
    bam = str(tmp_path / "in.bam"); fa = str(tmp_path / "ref.fa")
    bamio.write_bam(bam, [(c.name, c.length, c.reads)]); bamio.write_fasta(fa, [(c.name, c.ref)])
    p = subprocess.run([CLI, "coverage", bam, "-r", fa, "-L", "chrZ"], cwd=tmp_path, capture_output=True, text=True)
    assert p.returncode != 0 and "None of the specified contigs (chrZ) were found in the BAM file" in p.stderr


@pytest.mark.parametrize("case", ["unsorted", "truncated", "svg_collision_1_contig", "svg_collision_6_contigs"])
def test_cli_failures_exit_1_with_the_error(tmp_path, case):
    """Bad input files and unwritable outputs end in `Error: <message>` and exit code 1, whichever thread meets the failure
    (decoder: unsorted or truncated BAM; device thread: a directory where a coverage plot goes, while the decoder is done
    or still running).  With --progress the failure is also the last event, after Started."""
    cs = [synth.synth_short("chr1", 120_000, seed=44)]
    if case == "svg_collision_6_contigs":
        cs += [synth.synth_short(f"chr{i}", 60_000, seed=44 + i) for i in range(2, 7)]
    contigs = [(c.name, c.length, c.reads) for c in cs]
    if case == "unsorted":                                   # the second half of the records in reverse order
        n = cs[0].reads.n
        contigs = [(cs[0].name, cs[0].length, cs[0].reads.select(np.concatenate([np.arange(n // 2), np.arange(n - 1, n // 2 - 1, -1)])))]
        want = "Error processing contig: records are not coordinate sorted"
    elif case == "truncated":
        want = "truncated"
    else:
        (tmp_path / "chr1_coverage.svg").mkdir()
        want = f"Error processing contig: cannot create {tmp_path / 'chr1_coverage.svg'}"
    bam = str(tmp_path / "in.bam"); fa = str(tmp_path / "ref.fa")
    bamio.write_bam(bam, contigs); bamio.write_fasta(fa, [(c.name, c.ref) for c in cs])
    if case == "truncated":
        raw = open(bam, "rb").read()
        open(bam, "wb").write(raw[: len(raw) * 2 // 3])
    for extra in ([], ["--progress"]):
        p = subprocess.run([CLI, "coverage", bam, "-r", fa, "-o", str(tmp_path / "out.bed"), *extra], cwd=tmp_path,
                           capture_output=True, text=True, timeout=120)
        assert p.returncode == 1, p.stderr[-2000:]
        last = p.stderr.splitlines()[-1]
        assert last.startswith("Error: ") and want in last, p.stderr[-2000:]
        events = [json.loads(line) for line in p.stderr.splitlines() if line.startswith("{")]
        if extra:
            assert events[0] == {"Started": {"task": "Coverage Analysis"}}
            assert events[-1] == {"Error": {"task": "Coverage Analysis", "error": last[len("Error: "):]}}
        else:
            assert events == []


def test_cli_report_outputs_match_the_python_mirror(tmp_path):
    """Rows N2-N4: SVG plots from the device bins, HTML page, platform inference -- C++ (report_writer.hpp) against the
    Python mirror (report.py / bam_stats.py) fed with the ORACLE's bins and the JSON the CLI wrote."""
    from decodingustools_b200 import report
    cs = [synth.synth_short("chr1", 90_000, seed=51), synth.synth_short("chr2", 40_000, seed=52), synth.synth_short("chrM", 16_569, seed=53, depth=200.0)]
    contigs = [(c.name, tid, c.length, c.ref, c.reads) for tid, c in enumerate(cs)]
    bam = str(tmp_path / "in.bam"); fa = str(tmp_path / "ref.fa")
    bamio.write_bam(bam, [(n, l, r) for n, _, l, _, r in contigs], qname_fn=lambda contig, i: f"A00123:7:HFLOWCELLX:1:1101:{contig}:{i}")
    bamio.write_fasta(fa, [(n, ref) for n, _, _, ref, _ in contigs])
    tdir = tmp_path / "tpl"; tdir.mkdir()
    (tdir / "report_header.html").write_text("<html><!-- custom header -->\n"); (tdir / "report_footer.html").write_text("<!-- custom footer --></html>")
    for extra, head, foot in (([], report.DEFAULT_REPORT_HEADER, report.DEFAULT_REPORT_FOOTER),
                              (["--report-templates", str(tdir)], "<html><!-- custom header -->\n", "<!-- custom footer --></html>")):
        p = subprocess.run([CLI, "coverage", bam, "-r", fa, "-o", "out.bed", *extra], cwd=tmp_path, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr
        js = json.load(open(tmp_path / "summary.json"))
        o = run_oracle(contigs, CallableOptions())
        assert open(tmp_path / "out.bed", "rb").read() == o.bed()
        for oc in o.contigs:
            path = tmp_path / f"{oc.name}_coverage.svg"
            assert path.exists() == (oc.bins is not None)
            if oc.bins is not None:
                assert path.read_text() == report.render_coverage_svg(oc.name, oc.length, oc.stride, oc.bins), oc.name
        assert js["export"]["summary"]["sequencing_platform"] == "NovaSeq" and js["export"]["summary"]["read_length"] == 150
        assert js["files"]["coverage_plots"] == [f"{oc.name}_coverage.svg" for oc in o.contigs if oc.bins is not None]
        assert (tmp_path / "summary.json").read_text() == report.render_summary_json(js["export"], "out.bed", "summary.html", js["files"]["coverage_plots"])
        html = (tmp_path / "summary.html").read_text()
        assert html == report.render_html_report(js["export"], header_html=head, footer_html=foot, plot_exists=lambda q: (tmp_path / q).exists())
        assert html.count("<figure") == sum(oc.bins is not None for oc in o.contigs) > 0


def test_cli_progress_events_follow_the_reference_api(tmp_path):
    """--progress: the reference API's ProgressEvent stream (api/mod.rs:12-18) as serde-style JSON lines on stderr."""
    cs = [synth.synth_short("chr1", 30_000, seed=51), synth.synth_short("chr2", 20_000, seed=52)]
    bam = str(tmp_path / "in.bam"); fa = str(tmp_path / "ref.fa")
    bamio.write_bam(bam, [(c.name, c.length, c.reads) for c in cs], index=False, block=0xFF00)
    bamio.write_fasta(fa, [(c.name, c.ref) for c in cs])
    p = subprocess.run([CLI, "coverage", bam, "-r", fa, "-o", str(tmp_path / "out.bed"), "--progress"], cwd=tmp_path,
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    events = [json.loads(line) for line in p.stderr.splitlines() if line.startswith("{")]
    task = {"task": "Coverage Analysis"}
    assert events[0] == {"Started": task} and events[-1] == {"Completed": task}
    assert events[1:-1] == [{"Progress": {**task, "current": i + 1, "total": 2}} for i in range(2)]
