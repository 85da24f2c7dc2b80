"""Pins the CPU restatement (oracle/port) -- and the product's host readers/emitters it shares -- against the compiled
reference binary on seeded synthetic inputs of a few thousand reads (every output file, both passes, split pieces).
Where oracle/_ref/lr2rmats is built the reference runs alongside; elsewhere its outputs are known by their digests
(the pin_* entries of tests/golden/ref_digests.json)."""
import os

import numpy as np
import pytest

from lr2rmats_b200 import cabi, synth
from tests import oracle_port as op


@pytest.fixture(scope="module")
def workdir(tmp_path_factory):
    d = tmp_path_factory.mktemp("pin")
    anno = synth.make_annotation(700, n_chrom=3, seed=31)
    rr = synth.make_rrna(anno, 20, seed=32)
    synth.write_gtf(d / "anno.gtf", anno); synth.write_rm_gtf(d / "rm.gtf", rr, anno.chrom_names)
    for name, ont, seed, n in (("iso", False, 33, 5000), ("ont", True, 34, 1200)):
        r = synth.make_reads(anno, n, seed=seed, ont=ont, reject_frac=0.2, rrna=rr, quirk_frac=0.03)
        synth.write_sam(d / f"{name}.sam", r, with_seq=True)
        ex = op.bam2gtf(r.soa(), cabi.ExonParams.default())
        sj = synth.make_sj((ex["tid"], ex["exon_off"], ex["exon_start"], ex["exon_end"]), 0.7, seed=5)
        synth.write_sj(d / f"{name}.sj.tab", sj, anno.chrom_names)
    op.check_inputs("pin_inputs", {fn: d / fn for fn in sorted(os.listdir(d))})
    return d


def run_one(workdir, tag, who, binary, args, stdout_name):
    o = workdir / f"{tag}_{who}"
    o.mkdir(exist_ok=True)
    a = [x.replace("@", str(o) + "/") for x in args]
    op.run_bin(binary, a, str(o / stdout_name) if stdout_name else None)
    return {fn: op.digest(o / fn) for fn in sorted(os.listdir(o))}


def run_both(workdir, tag, args, stdout_name=None):
    """Every output file of the port equals the reference's (a .bam after decompression: the deflate bytes depend on zlib)."""
    got = run_one(workdir, tag, "port", op.PORT_BIN, args, stdout_name)
    ref = run_one(workdir, tag, "ref", op.REF_BIN, args, stdout_name) if op.have_ref_bin() else None
    want = op.stored_digests(f"pin_{tag}", ref)
    if ref is not None:
        assert ref == want, f"{tag}: the reference's outputs differ from the stored digests"
    assert sorted(got) == sorted(want)
    for fn in want:
        assert got[fn] == want[fn], f"{tag}: {fn} differs"
    return sorted(want)


ALL = ["-A", "@detail.txt", "-y", "@summary.txt", "-E", "@bed", "-a", "@bam.gtf", "-k", "@known.gtf", "-v", "@novel.gtf", "-u", "@unrecog.gtf", "-o", "@updated.gtf"]


@pytest.mark.parametrize("which", ["iso", "ont"])
def test_filter_bam2gtf_unique(workdir, which):
    sam = str(workdir / f"{which}.sam")
    run_both(workdir, f"{which}_filter", ["filter", "-r", str(workdir / "rm.gtf"), sam], "out.bam")
    run_both(workdir, f"{which}_b2g", ["bam2gtf", sam], "out.gtf")
    run_both(workdir, f"{which}_uniq", ["unique-gtf", sam], "out.gtf")


@pytest.mark.parametrize("which", ["iso", "ont"])
@pytest.mark.parametrize("level", ["1", "3", "5"])
def test_update_pass1(workdir, which, level):
    run_both(workdir, f"{which}_p1_{level}", ["update-gtf", "-l", level, str(workdir / f"{which}.sam"), str(workdir / "anno.gtf")] + ALL)


@pytest.mark.parametrize("which", ["iso", "ont"])
@pytest.mark.parametrize("extra", [["-s"], [], ["-s", "-d", "5", "-J", "2"], ["-s", "-c", "-M", "x"]])
def test_update_pass2(workdir, which, extra):
    tag = f"{which}_p2_" + "".join(e.strip("-") for e in extra)
    run_both(workdir, tag, ["update-gtf"] + extra + ["-l", "3", "-j", str(workdir / f"{which}.sj.tab"), str(workdir / f"{which}.sam"), str(workdir / "anno.gtf")] + ALL)


def test_gtf_input_mode(workdir):
    """-m g: the novel GTF of pass 1 fed back as input (Snakefile:189-192 uses unique-gtf -m g)."""
    sam = str(workdir / "iso.sam")
    run_both(workdir, "gin", ["update-gtf", "-l", "3", sam, str(workdir / "anno.gtf")], "novel.gtf")
    novel = str(workdir / "gin_port" / "novel.gtf")                  # byte-equal to the reference's
    run_both(workdir, "gin_uniq", ["unique-gtf", "-m", "g", "-b", sam, novel], "out.gtf")
    run_both(workdir, "gin_upd", ["update-gtf", "-m", "g", "-b", sam, "-l", "5", novel, str(workdir / "anno.gtf")] + ALL)


@pytest.mark.parametrize("which", ["iso", "ont"])
def test_bam2sj(workdir, which, tmp_path):
    """bam2sj on a few thousand paired records with NH tags (and some without): port == reference binary, default and -i; the single-end
    original gives the header only (read_type is PAIR_T whatever the options say, parse_bam.c:76,997)."""
    anno = synth.make_annotation(700, n_chrom=3, seed=31)
    r = synth.make_reads(anno, 3000 if which == "iso" else 800, seed=35, ont=(which == "ont"), reject_frac=0.1)
    rng = np.random.default_rng(36)
    r.flag = (r.flag | np.where(rng.random(r.n) < 0.8, np.uint16(3), np.uint16(0))).astype(np.uint16)     # 80 % proper pairs
    nh = rng.choice([0, 1, 1, 1, 2, 5], r.n)
    sam = tmp_path / "paired.sam"
    synth.write_sam(sam, r, with_seq=False, nh=nh)
    op.check_inputs(f"pin_{which}_sj_inputs", {"paired.sam": sam})
    names = run_both(workdir, f"{which}_sj", ["bam2sj", str(sam)], "out.sj")
    run_both(workdir, f"{which}_sj_i", ["bam2sj", "-i", "300", str(sam)], "out.sj")
    assert sum(1 for _ in open(workdir / f"{which}_sj_port" / "out.sj")) > 50          # the outputs equal the reference's
    run_both(workdir, f"{which}_sj_se", ["bam2sj", str(workdir / f"{which}.sam")], "out.sj")
    assert sum(1 for _ in open(workdir / f"{which}_sj_se_port" / "out.sj")) == 4


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_sort_gtf_fuzz(seed, tmp_path):
    """`sort-gtf` (host tagging + stable three-key sort; the port CLI sorts with std::stable_sort where the product uses the device) against
    the reference's own script on random concatenations: shuffled transcripts of known / unknown chromosomes, equal keys, foreign feature
    lines, comments, blanks instead of tabs, short lines, leading zeros."""
    import random
    import subprocess
    rnd = random.Random(seed)
    chroms = ["chr1", "chr2", "chr10", "chrX", "chrM", "chrUn_a", "scaf7", "chr22", "KI270", "chrY"]
    blocks = []
    for t in range(rnd.randint(40, 120)):
        ch = rnd.choice(chroms); s = rnd.choice([rnd.randint(1, 50), rnd.randint(1, 100000)]); e = s + rnd.randint(0, 5000)
        ss = ("%05d" % s) if rnd.random() < 0.1 else str(s)
        sep = " " if rnd.random() < 0.05 else "\t"
        lines = [sep.join([ch, "src", "transcript", ss, str(e), ".", rnd.choice("+-"), "."]) + f'\tgene_id "G{t}"; transcript_id "T{t}";']
        for x in range(rnd.randint(0, 4)):
            kind = rnd.choice(["exon", "exon", "exon", "CDS", "start_codon", "transcript_part"])
            cols = [ch, "src", kind, str(s + x), str(e - x), ".", "+", ".", f'gene_id "G{t}"; transcript_id "T{t}"; exon_number "{x}";']
            if rnd.random() < 0.1: cols = cols[:rnd.randint(5, 8)]
            if rnd.random() < 0.05: cols.append("extra")
            lines.append("\t".join(cols))
        if rnd.random() < 0.1: lines.insert(rnd.randint(0, len(lines)), "# comment " + str(t))
        if rnd.random() < 0.05: lines.append("")
        blocks.append(lines)
    rnd.shuffle(blocks)
    head = ["chr5\tsrc\texon\t10\t20\t.\t+\t.\tgene_id \"pre\";"] if seed % 2 else []
    text = "\n".join(head + [ln for b in blocks for ln in b]) + "\n"
    (tmp_path / "in.gtf").write_text(text)
    op.check_inputs(f"pin_sort_gtf_{seed}_inputs", {"in.gtf": tmp_path / "in.gtf"})
    want = op.ref_digests(f"pin_sort_gtf_{seed}", lambda: subprocess.run(["bash", op.REF_SORT_SCRIPT, str(tmp_path / "in.gtf"), str(tmp_path / "ref.gtf")],
                                                                          check=True, env=dict(os.environ, LC_ALL="C")), {"sorted.gtf": tmp_path / "ref.gtf"},
                          available=os.path.isfile(op.REF_SORT_SCRIPT))
    op.run_bin(op.PORT_BIN, ["sort-gtf", str(tmp_path / "in.gtf"), str(tmp_path / "port.gtf")])
    assert op.digest(tmp_path / "port.gtf") == want["sorted.gtf"]
