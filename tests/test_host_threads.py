"""SURVEY row f-1: the multi-threaded host decode / encode (BGZF inflate by block, BAM records and SAM lines by chunk,
BGZF deflate by block group) gives the same bytes as the single-threaded code and as the reference binary (htslib) on
inputs large enough to be cut into several chunks.  The port CLI (oracle/_ref/lr2rmats_port) runs the product's own
readers and writers, so no GPU is needed here.  Where oracle/_ref/lr2rmats is built the reference runs alongside; elsewhere its
outputs are known by their digests (the threads_* entries of tests/golden/ref_digests.json), and the BAM inputs that the reference
would write are written by the port instead (same records, the product's BGZF blocks)."""
import os
import subprocess
import time

import pytest

from lr2rmats_b200 import synth
from tests import oracle_port as op



def run(binary, args, out, threads=None):
    env = dict(os.environ)
    if threads is not None:
        env["LRB_THREADS"] = str(threads)
    t0 = time.perf_counter()
    with open(out, "wb") as f:
        subprocess.run([binary] + args, stdout=f, stderr=subprocess.DEVNULL, check=True, env=env)
    return time.perf_counter() - t0


def filtered_bam(big):
    """filter's BAM of the big input: the reference's (htslib-written BGZF) where it is built, else the port's (same records)."""
    have = op.have_ref_bin()
    out = big / ("f_ref.bam" if have else "f_port.bam")
    if not os.path.exists(out):
        run(op.REF_BIN if have else op.PORT_BIN, ["filter", "-r", str(big / "rm.gtf"), str(big / "in.sam")], out)
    return out


@pytest.fixture(scope="module")
def big(tmp_path_factory):
    d = tmp_path_factory.mktemp("mt")
    anno = synth.make_annotation(3000, n_chrom=6, seed=41)
    rr = synth.make_rrna(anno, 30, seed=42)
    reads = synth.make_reads(anno, 40000, seed=43, ont=False, reject_frac=0.2, rrna=rr, quirk_frac=0.02)
    synth.write_sam(d / "in.sam", reads, with_seq=True)
    synth.write_rm_gtf(d / "rm.gtf", rr, anno.chrom_names)
    assert os.path.getsize(d / "in.sam") > 8 << 20          # several SAM chunks, > 100 BGZF blocks
    op.check_inputs("threads_inputs", {"in.sam": d / "in.sam", "rm.gtf": d / "rm.gtf"})
    return d


def test_sam_decode_and_bam_encode_threads(big):
    sam = str(big / "in.sam")
    a = ["filter", "-r", str(big / "rm.gtf"), sam]
    want = op.ref_digests("threads_sam", lambda: (run(op.REF_BIN, a, big / "f_ref.bam"), run(op.REF_BIN, ["bam2gtf", sam], big / "g_sam_ref.gtf")),
                          {"filter.bam": big / "f_ref.bam", "bam2gtf.gtf": big / "g_sam_ref.gtf"})
    run(op.PORT_BIN, a, big / "f_t1.bam", threads=1)
    run(op.PORT_BIN, a, big / "f_t8.bam", threads=8)
    assert open(big / "f_t1.bam", "rb").read() == open(big / "f_t8.bam", "rb").read()          # same BGZF blocks, same bytes
    assert op.digest(big / "f_t8.bam") == want["filter.bam"]
    for t in (1, 8):
        run(op.PORT_BIN, ["bam2gtf", sam], big / f"g_sam_t{t}.gtf", threads=t)
    got = open(big / "g_sam_t1.gtf", "rb").read()
    assert got == open(big / "g_sam_t8.gtf", "rb").read() and op.digest(big / "g_sam_t1.gtf") == want["bam2gtf.gtf"] and len(got) > 1 << 20


def test_bam_decode_threads(big):
    src = filtered_bam(big)                                   # htslib-written BGZF in (where the reference is built), decoded by 1, 3 and 8 threads
    want = op.ref_digests("threads_bam", lambda: (run(op.REF_BIN, ["bam2gtf", str(src)], big / "g_bam_ref.gtf"), run(op.REF_BIN, ["filter", str(src)], big / "ff_ref.bam")),
                          {"bam2gtf.gtf": big / "g_bam_ref.gtf", "filter.bam": big / "ff_ref.bam"})
    for t in (1, 3, 8):
        run(op.PORT_BIN, ["bam2gtf", str(src)], big / f"g_bam_t{t}.gtf", threads=t)
        assert op.digest(big / f"g_bam_t{t}.gtf") == want["bam2gtf.gtf"]
    assert os.path.getsize(big / "g_bam_t1.gtf") > 1 << 20
    # filter on BAM input re-emits the raw records: byte-equal streams again
    run(op.PORT_BIN, ["filter", str(src)], big / "ff_t8.bam", threads=8)
    assert op.digest(big / "ff_t8.bam") == want["filter.bam"]


def test_truncated_bgzf_and_malformed_sam(big, tmp_path):
    """A BAM cut inside a block and a SAM with a broken line deep in the file end the input there, on any thread count."""
    raw = open(filtered_bam(big), "rb").read()
    open(tmp_path / "cut.bam", "wb").write(raw[: len(raw) * 2 // 3])
    lines = open(big / "in.sam", "rb").read().split(b"\n")
    k = len(lines) * 3 // 4
    lines[k] = lines[k].replace(b"\t", b" ", 3)
    open(tmp_path / "bad.sam", "wb").write(b"\n".join(lines))
    for name in ("cut.bam", "bad.sam"):
        outs = []
        for t in (1, 8):
            run(op.PORT_BIN, ["bam2gtf", str(tmp_path / name)], tmp_path / f"{name}.t{t}.gtf", threads=t)
            outs.append(open(tmp_path / f"{name}.t{t}.gtf", "rb").read())
        assert outs[0] == outs[1] and len(outs[0]) > 1 << 19


def test_bgzf_crc_mismatch_is_read_like_the_reference(big, tmp_path):
    """A block whose CRC field is damaged but whose deflate stream is intact: the reference's htslib (1.3) never looks at the CRC and reads
    the file to its end; the product's decoder must give the same records (it only warns), on any thread count."""
    d = bytearray(open(filtered_bam(big), "rb").read())
    p, blocks = 0, []
    while p + 18 <= len(d):
        bsize = (d[p + 16] | (d[p + 17] << 8)) + 1
        blocks.append((p, bsize)); p += bsize
    assert len(blocks) > 10
    for k in (3, len(blocks) // 2):
        d[blocks[k][0] + blocks[k][1] - 8] ^= 0xFF               # first byte of the block's CRC32
    open(tmp_path / "crc.bam", "wb").write(d)
    want = op.ref_digests("threads_crc", lambda: run(op.REF_BIN, ["bam2gtf", str(tmp_path / "crc.bam")], tmp_path / "ref.gtf"), {"bam2gtf.gtf": tmp_path / "ref.gtf"})
    for t in (1, 8):
        run(op.PORT_BIN, ["bam2gtf", str(tmp_path / "crc.bam")], tmp_path / f"port.t{t}.gtf", threads=t)
        assert op.digest(tmp_path / f"port.t{t}.gtf") == want["bam2gtf.gtf"]
    assert os.path.getsize(tmp_path / "port.t1.gtf") > 1 << 19


def test_emitters_threads(big, tmp_path):
    """Row f-2: every text output of update-gtf / unique-gtf formatted by 8 threads == 1 thread == the reference's printers."""
    from lr2rmats_b200 import cabi
    anno = synth.make_annotation(3000, n_chrom=6, seed=41)
    synth.write_gtf(tmp_path / "anno.gtf", anno)
    files = ["detail.txt", "summary.txt", "bed", "bam.gtf", "known.gtf", "novel.gtf", "unrecog.gtf", "updated.gtf"]
    flags = ["-A", "-y", "-E", "-a", "-k", "-v", "-u", "-o"]
    op.check_inputs("threads_anno_inputs", {"anno.gtf": tmp_path / "anno.gtf"})

    def emit(who, binary, t):
        d = tmp_path / who; d.mkdir()
        a = ["update-gtf", "-l", "5", str(big / "in.sam"), str(tmp_path / "anno.gtf")]
        for fl, fn in zip(flags, files):
            a += [fl, str(d / fn)]
        run(binary, a, d / "stdout", threads=t)
        run(binary, ["unique-gtf", str(big / "in.sam")], d / "uniq.gtf", threads=t)

    want = op.ref_digests("threads_emitters", lambda: emit("ref", op.REF_BIN, None), {fn: tmp_path / "ref" / fn for fn in files + ["uniq.gtf"]})
    outs = {}
    for who, t in (("t1", 1), ("t8", 8)):
        emit(who, op.PORT_BIN, t)
        outs[who] = {fn: open(tmp_path / who / fn, "rb").read() for fn in files + ["uniq.gtf"]}
    for fn in files + ["uniq.gtf"]:
        assert outs["t1"][fn] == outs["t8"][fn] and op.digest(tmp_path / "t1" / fn) == want[fn], fn
    assert len(outs["t1"]["updated.gtf"]) > 1 << 20 and len(outs["t1"]["detail.txt"]) > 1 << 20 and len(outs["t1"]["known.gtf"]) > 1 << 16


@pytest.mark.parametrize("quirk", ["plain", "comments_cds", "blank_separated", "long_line", "no_names"])
def test_gtf_reader_threads(big, tmp_path, quirk):
    """The all-threads annotation reader takes plain files only; anything else must fall back to the reference's own parsing
    (fgets 1024 + sscanf state, SURVEY Q7/Q8) -- the outputs equal the reference binary's either way."""
    anno = synth.make_annotation(3000, n_chrom=6, seed=41)
    synth.write_gtf(tmp_path / "anno.gtf", anno)
    lines = open(tmp_path / "anno.gtf").read().split("\n")
    k = len(lines) // 2
    while "\texon\t" not in lines[k]:
        k += 1
    if quirk == "comments_cds":
        lines[k:k] = ["# a comment", lines[k].replace("\texon\t", "\tCDS\t"), "#another"]
    elif quirk == "blank_separated":
        lines[k] = lines[k].replace("\t", " ", 4)
    elif quirk == "long_line":
        lines[k] = lines[k] + " note \"" + "ab " * 400 + "\";"          # tokens stay below the reference's ref[100] / type[20] buffers
    elif quirk == "no_names":
        lines[k] = lines[k].split("gene_name")[0].rstrip()
    open(tmp_path / "anno.gtf", "w").write("\n".join(lines))
    op.check_inputs(f"threads_gtf_{quirk}_inputs", {"anno.gtf": tmp_path / "anno.gtf"})
    files = ("updated.gtf", "summary.txt", "known.gtf")

    def update(name, binary, env):
        d = tmp_path / name; d.mkdir()
        e = dict(os.environ); e.update(env)
        with open(d / "updated.gtf", "wb") as f:
            p = subprocess.run([binary, "update-gtf", "-l", "5", str(big / "in.sam"), str(tmp_path / "anno.gtf"), "-y", str(d / "summary.txt"), "-k", str(d / "known.gtf")],
                               stdout=f, stderr=subprocess.DEVNULL, env=e)
        assert p.returncode == 0, name
        return d

    want = op.ref_digests(f"threads_gtf_{quirk}", lambda: update("ref", op.REF_BIN, {}), {fn: tmp_path / "ref" / fn for fn in files})
    for name, env in (("t8", {"LRB_THREADS": "8"}), ("seq", {"LRB_GTF_SEQUENTIAL": "1"})):
        d = update(name, op.PORT_BIN, env)
        assert {fn: op.digest(d / fn) for fn in files} == want, name
    assert os.path.getsize(tmp_path / "t8" / "updated.gtf") > 1 << 20


@pytest.mark.parametrize("quirk", ["plain", "short_line", "unknown_chrom_blank"])
def test_sj_reader_threads(big, tmp_path, quirk):
    """SJ.out.tab through the all-threads reader (plain files) or the reference's sscanf loop (anything else): same
    junction support, same chromosome-id extension (gtf.c:389-449)."""
    from lr2rmats_b200 import cabi
    anno = synth.make_annotation(3000, n_chrom=6, seed=41)
    rr = synth.make_rrna(anno, 30, seed=42)
    reads = synth.make_reads(anno, 40000, seed=43, ont=False, reject_frac=0.2, rrna=rr, quirk_frac=0.02)
    ex = op.bam2gtf(reads.soa(), cabi.ExonParams.default())
    sj = synth.make_sj((ex["tid"], ex["exon_off"], ex["exon_start"], ex["exon_end"]), 0.7, seed=5)
    synth.write_gtf(tmp_path / "anno.gtf", anno); synth.write_sj(tmp_path / "sj.tab", sj, anno.chrom_names)
    lines = open(tmp_path / "sj.tab").read().split("\n")
    assert len(lines) > 20000
    k = len(lines) // 2
    if quirk == "short_line":
        lines[k] = "\t".join(lines[k].split("\t")[:5])               # later columns keep the previous line's values
    elif quirk == "unknown_chrom_blank":
        lines[k] = lines[k].replace("\t", " ", 2); lines[k + 1] = "chrUn_x\t" + lines[k + 1].split("\t", 1)[1]
    open(tmp_path / "sj.tab", "w").write("\n".join(lines))
    op.check_inputs(f"threads_sj_{quirk}_inputs", {"anno.gtf": tmp_path / "anno.gtf", "sj.tab": tmp_path / "sj.tab"})
    files = ("updated.gtf", "summary.txt", "detail.txt")

    def update(name, binary, env):
        d = tmp_path / name; d.mkdir()
        e = dict(os.environ); e.update(env)
        with open(d / "updated.gtf", "wb") as f:
            p = subprocess.run([binary, "update-gtf", "-s", "-l", "3", "-j", str(tmp_path / "sj.tab"), str(big / "in.sam"), str(tmp_path / "anno.gtf"),
                                "-y", str(d / "summary.txt"), "-A", str(d / "detail.txt")], stdout=f, stderr=subprocess.DEVNULL, env=e)
        assert p.returncode == 0, name
        return d

    want = op.ref_digests(f"threads_sj_{quirk}", lambda: update("ref", op.REF_BIN, {}), {fn: tmp_path / "ref" / fn for fn in files})
    for name, env in (("t8", {"LRB_THREADS": "8"}), ("seq", {"LRB_GTF_SEQUENTIAL": "1"})):
        d = update(name, op.PORT_BIN, env)
        assert {fn: op.digest(d / fn) for fn in files} == want, name
    assert os.path.getsize(tmp_path / "t8" / "updated.gtf") > 1 << 20


def test_io_bench_tool_digest(big):
    """lrb-io-bench (the host decode / encode timer of DESIGN 6.4) decodes to the same SoA batch on 1 and 8 threads."""
    import json
    tool = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lr2rmats_b200", "host", "lrb-io-bench")
    if not os.path.exists(tool):
        pytest.skip("lrb-io-bench not built")
    outs = []
    for t in (1, 8):
        env = dict(os.environ, LRB_THREADS=str(t))
        p = subprocess.run([tool, str(big / "in.sam"), str(big / f"iob_t{t}.bam")], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, check=True, env=env)
        outs.append(json.loads(p.stdout))
    assert outs[0]["digest"] == outs[1]["digest"] and outs[0]["records"] == outs[1]["records"] > 40000
    assert outs[0]["threads"] == 1 and outs[1]["threads"] == 8
    assert open(big / "iob_t1.bam", "rb").read() == open(big / "iob_t8.bam", "rb").read()
