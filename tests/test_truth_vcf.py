"""SIMUSCOP_TRUTH_VCF=1: the per-sample truth VCF (DESIGN.md section 10) against the haplotype strings of the plan dumps, which
test_host_plan_matches_golden_hashes pins to the instrumented reference's.  An independent applier rebuilds every haplotype of
every segment from the FASTA and the VCF records; the plans must not move when the file is written."""
import glob
import hashlib
import os
import re
import struct
import subprocess

import numpy as np
import pytest

import helpers
from simuscop_b200 import planfile, synth
from simuscop_b200.paths import SIMUREADS

ROUND_TRIP = ["pe_variants", "pe_ploidy3", "se_ploidy1", "se_tumor", "pe_iupac", "pe_wes"]
EDGE_SEEDS = [s for kind, s in helpers.EDGE_CASES if kind == "variation"]


def abbr(name):
    """abbr_chr: the chr-stripped name the variation files, read names and plan dumps use."""
    for p in ("chrom", "chr"):
        i = name.find(p)
        if i >= 0:
            return name[i + len(p):]
    return name


def read_fasta(path):
    """[(first word of the header line, upper-cased sequence)] in file order."""
    out = []
    with open(path) as f:
        for rec in f.read().split(">")[1:]:
            head, body = rec.split("\n", 1)
            out.append((head.split()[0], body.replace("\n", "").upper()))
    return out


def plan_units(path):
    """The haplotype strings of a plan dump: [(popu, chr, [dict(start, end, CN, haps)])] in dump order."""
    planfile.read_plan(path)                      # validates the whole file
    data = open(path, "rb").read()
    off, units = 8, []
    while off < len(data):
        tag, n = struct.unpack_from("<iq", data, off)
        off += 12
        body = data[off:off + n]
        off += n
        if tag == 2:
            pl, cl = struct.unpack_from("<2i", body, 0)
            units.append((body[8:8 + pl].decode(), body[8 + pl:8 + pl + cl].decode(), []))
        elif tag == 3:
            _, CN, start, end, _, _, _, ploidy = struct.unpack_from("<2i4q2i", body, 0)
            lens = struct.unpack_from("<%dq" % ploidy, body, 48)
            o, haps = 48 + 8 * ploidy, []
            for L in lens:
                haps.append(body[o:o + L].decode("latin-1"))
                o += L
            units[-1][2].append(dict(start=start, end=end, CN=CN, haps=haps))
        elif tag == 9:
            break
    return units


def parse_vcf(path):
    meta, cols, recs = [], None, []
    for line in open(path).read().splitlines():
        if line.startswith("##"):
            meta.append(line)
        elif line.startswith("#"):
            cols = line[1:].split("\t")
        else:
            f = line.split("\t")
            info = dict(kv.split("=", 1) for kv in f[7].split(";"))
            recs.append(dict(chrom=f[0], pos=int(f[1]), ref=f[3], alt=f[4], info=info, fmt=f[8].split(":"), samples=f[9:], line=line))
    return meta, cols, recs


def locus(r):
    """The first changed reference base (the anchor of an insertion or SNV): the segment a record belongs to."""
    if len(r["ref"]) == 1:
        return r["pos"]
    return 1 if right_anchored(r) else r["pos"] + 1


def right_anchored(r):
    """A change in front of chromosome position 1 carries the base after it (VCF 4.2, section 1.6.1)."""
    return r["pos"] == 1 and r["ref"][0] != r["alt"][0]


def apply_copy(slice_, start, recs):
    """The upper-cased reference slice [start, start + len) with the records one copy holds applied."""
    base = list(slice_)
    n = len(base)
    gone = [False] * n
    ins = [""] * (n + 1)
    for r in recs:
        ref, alt, pos = r["ref"], r["alt"], r["pos"]
        if len(ref) == 1 and len(alt) == 1:
            base[pos - start] = alt
            continue
        if right_anchored(r):
            d0, e, lit = 1, pos + len(ref) - 1, alt[:-1]
        else:
            d0, e, lit = pos + 1, pos + len(ref), alt[1:]
        for p in range(d0, e):
            assert 0 <= p - start < n, (r["line"], start)
            gone[p - start] = True
        assert ins[e - start] == "", "two changes in one gap: %s" % r["line"]
        ins[e - start] = lit
    return "".join(ins[i] + ("" if gone[i] else base[i]) for i in range(n)) + ins[n]


def run_plan_only(scn, tag, truth):
    d = scn["dir"]
    out = os.path.join(d, "out_" + tag)
    cfg = os.path.join(d, "cfg_%s.txt" % tag)
    synth.write_config(cfg, output=out, **scn["kw"])
    for f in glob.glob(os.path.join(d, "plan_%s.*" % tag)) + glob.glob(os.path.join(out, "*.truth.vcf")):
        os.remove(f)
    env = dict(os.environ, SIMUSCOP_SEED=str(scn["seed"]), SIMUSCOP_DUMP_PLAN=os.path.join(d, "plan_" + tag), SIMUSCOP_PLAN_ONLY="1")
    env.pop("SIMUSCOP_TRUTH_VCF", None)
    if truth:
        env["SIMUSCOP_TRUTH_VCF"] = "1"
    r = subprocess.run([SIMUREADS, cfg], env=env, capture_output=True, text=True, timeout=600)
    plans = sorted(glob.glob(os.path.join(d, "plan_%s.*.plan" % tag)), key=lambda p: int(p.split(".")[-2]))
    return plans, out, r


def abundance_rows(scn):
    if not scn["kw"].get("abundance"):
        return []
    return [l.split("\t") for l in open(scn["kw"]["abundance"]).read().splitlines() if l]


def stems(scn):
    """File-name stem of every output sample (ssh_sample_stem): the first population alone without abundance rows."""
    names = scn["kw"]["name"].split(",")
    rows = abundance_rows(scn)
    return ["+".join("%s_%.3f" % (n, float(p)) for n, p in zip(names, row)) for row in rows] if rows else [names[0]]


def props(scn):
    return [[float(x) for x in row] for row in abundance_rows(scn)] or [[1.0]]


def cnv_lines(scn):
    """(popu, abbreviated chr, spos, epos, cn, mcn) of every 'c' record of the variation file."""
    out = []
    if scn["kw"].get("variation"):
        for l in open(scn["kw"]["variation"]).read().splitlines():
            f = l.split("\t")
            if f[0] == "c":
                out.append((f[1], abbr(f[2]), int(f[3]), int(f[4]), int(f[5]), int(f[6])))
    return out


def check_truth(scn, plans, vcfs):
    """Every check of a truth file against its plan dump, FASTA and sample: see the module docstring."""
    fasta = read_fasta(scn["kw"]["ref"])
    seq = {abbr(n): s for n, s in fasta}
    order = {n: i for i, (n, _) in enumerate(fasta)}
    pops = scn["kw"]["name"].split(",")
    ploidy = int(scn["kw"].get("ploidy", 2))
    cnvs = cnv_lines(scn)
    bodies = []
    for si, (plan, vcf) in enumerate(zip(plans, vcfs)):
        meta, cols, recs = parse_vcf(vcf)
        # header
        assert meta[0] == "##fileformat=VCFv4.2"
        assert "##reference=" + scn["kw"]["ref"] in meta
        assert [m for m in meta if m.startswith("##contig")] == ["##contig=<ID=%s,length=%d>" % (n, len(s)) for n, s in fasta]
        for tag in ("INFO=<ID=EAF,", "INFO=<ID=END,", "FORMAT=<ID=GT,", "FORMAT=<ID=HCN,", "FORMAT=<ID=CN,", "FORMAT=<ID=MCN,", "ALT=<ID=CNV,"):
            assert any(m.startswith("##" + tag) for m in meta), tag
        assert cols == ["CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + pops
        # order, REF bases, one record per small variant
        keys = [(order[r["chrom"]], r["pos"], r["ref"], r["alt"]) for r in recs]
        assert keys == sorted(keys)
        small = [r for r in recs if r["alt"] != "<CNV>"]
        assert len({(r["chrom"], r["pos"], r["ref"], r["alt"]) for r in small}) == len(small)
        for r in recs:
            s = seq[abbr(r["chrom"])]
            want = s[r["pos"] - 1:r["pos"] - 1 + len(r["ref"])] if r["alt"] != "<CNV>" else s[r["pos"] - 1]
            assert r["ref"] == want, r["line"]
        units = plan_units(plan)
        segs = {(p, c): v for p, c, v in units}
        # small variants: GT ploidy, EAF, and the copies of every segment that holds the record's locus
        per_seg = {}            # (popu, chr, segment index) -> [(record, alleles of that segment's copies)]
        hcn_of = {}
        w = props(scn)[si]
        for r in small:
            assert r["fmt"] == ["GT", "HCN"]
            c = abbr(r["chrom"])
            num = den = 0.0
            any_alt = False
            for pi, p in enumerate(pops):
                v = segs.get((p, c), [])
                cover = [k for k, sg in enumerate(v) if sg["start"] <= locus(r) <= sg["end"]]
                if not cover:
                    assert r["samples"][pi] == ".", r["line"]
                    continue
                gt, hcn = r["samples"][pi].split(":")
                gt = [int(a) for a in gt.split("|")]
                hcn = [int(x) for x in hcn.split(",")]
                assert len(hcn) == ploidy * len(cover), r["line"]
                assert len(gt) == sum(hcn) == sum(v[k]["CN"] for k in cover), r["line"]
                at = 0
                for n, k in enumerate(cover):
                    h = hcn[n * ploidy:(n + 1) * ploidy]
                    assert hcn_of.setdefault((p, c, k), h) == h, r["line"]
                    per_seg.setdefault((p, c, k), []).append((r, gt[at:at + sum(h)]))
                    at += sum(h)
                num += w[pi] * sum(gt)
                den += w[pi] * len(gt)
                any_alt |= sum(gt) > 0
            assert any_alt, "a record no copy holds: " + r["line"]
            assert abs(float(r["info"]["EAF"]) - num / den) <= 1e-5 * max(1.0, num / den), r["line"]
        # CNV records: one per segment made from a 'c' record, its CN / MCN / HCN
        for r in recs:
            if r["alt"] != "<CNV>":
                continue
            assert r["fmt"] == ["CN", "MCN", "HCN"] and r["info"]["SVTYPE"] == "CNV"
            c, end = abbr(r["chrom"]), int(r["info"]["END"])
            [pi] = [i for i, x in enumerate(r["samples"]) if x != "."]
            p = pops[pi]
            cn, mcn, hcn = r["samples"][pi].split(":")
            hcn = [int(x) for x in hcn.split(",")]
            [k] = [k for k, sg in enumerate(segs[(p, c)]) if sg["start"] == r["pos"] and sg["end"] == end]
            sg = segs[(p, c)][k]
            assert int(cn) == sg["CN"] == sum(hcn) and len(hcn) == ploidy, r["line"]
            assert any(q == p and cc == c and a <= r["pos"] and end <= max(b, a) and n == int(cn) and m == int(mcn)
                       for q, cc, a, b, n, m in cnvs), r["line"]
            assert hcn_of.setdefault((p, c, k), hcn) == hcn, r["line"]
        assert sum(r["alt"] == "<CNV>" for r in recs) >= len({(q, cc, a) for q, cc, a, b, _, _ in cnvs
                                                              if cc in seq and a <= len(seq[cc]) and b >= a
                                                              and q in {u[0] for u in units}})
        # round trip: every haplotype of every segment, rebuilt copy by copy from the FASTA and the records
        for p, c, v in units:
            for k, sg in enumerate(v):
                slice_ = seq[c][sg["start"] - 1:sg["end"]]
                hcn = hcn_of.get((p, c, k), [1] * ploidy)
                assert sum(hcn) == sg["CN"], (p, c, sg["start"])
                at = 0
                for j in range(ploidy):
                    got = ""
                    for t in range(hcn[j]):
                        held = [r for r, al in per_seg.get((p, c, k), []) if al[at + t]]
                        got += apply_copy(slice_, sg["start"], held)
                    at += hcn[j]
                    assert got == sg["haps"][j], "%s %s:%d haplotype %d differs from the plan dump" % (p, c, sg["start"], j)
        bodies.append([r["line"] for r in recs])
    # files of different samples differ only in EAF
    strip = [[re.sub(r"EAF=[^;\t]*", "EAF", l) for l in b] for b in bodies]
    assert all(s == strip[0] for s in strip)
    return bodies


def truth_round_trip(scn):
    plans_off, out_off, r_off = run_plan_only(scn, "off", truth=False)
    assert not glob.glob(os.path.join(out_off, "*.truth.vcf"))
    plans, out, r = run_plan_only(scn, "truth", truth=True)
    last = [x.strip().split("\n")[-1].replace("_truth", "_off") for x in (r.stderr, r_off.stderr)]
    assert r.returncode == r_off.returncode and (r.returncode == 0 or last[0] == last[1]), r.stderr[-3000:]
    if r.returncode:            # an input the front end rejects: rejected the same way, before any truth file
        assert not glob.glob(os.path.join(out, "*.truth.vcf"))
        return []
    assert [helpers.read_file(a) for a in plans] == [helpers.read_file(b) for b in plans_off]
    vcfs = [os.path.join(out, s + ".truth.vcf") for s in stems(scn)]
    assert sorted(glob.glob(os.path.join(out, "*.truth.vcf"))) == sorted(vcfs)
    assert len(plans) == len(vcfs)
    return check_truth(scn, plans, vcfs)


@pytest.mark.parametrize("name", ROUND_TRIP)
def test_truth_rebuilds_plan_haplotypes(built, workdir, name):
    scn = helpers.build_scenario(name, os.path.join(workdir, "truth"))
    bodies = truth_round_trip(scn)
    if scn["kw"].get("variation") or scn["kw"].get("snp"):
        assert all(len(b) > 0 for b in bodies)


@pytest.mark.parametrize("seed", helpers.FUZZ_VARIATION_SEEDS)
def test_truth_rebuilds_random_variation_haplotypes(built, workdir, seed):
    truth_round_trip(helpers.build_random_variation_scenario(seed, os.path.join(workdir, "truth")))


@pytest.mark.parametrize("seed", EDGE_SEEDS)
def test_truth_rebuilds_edge_variation_haplotypes(built, workdir, seed):
    scn, _ = helpers.build_edge_variation_scenario(seed, os.path.join(workdir, "truth"))
    truth_round_trip(scn)


def test_truth_eaf_of_tumour_mixture(built, workdir):
    """se_tumor: four populations in two abundance rows; EAF = sum(props * ALT copies) / sum(props * copies)."""
    scn = helpers.build_scenario("se_tumor", os.path.join(workdir, "truth_eaf"))
    a, b = truth_round_trip(scn)
    assert len(a) == len(b) and a != b
    pure = [l for l in a if "<CNV>" not in l]
    # the first row is clone1 alone: a change clone1 lacks has EAF 0, one on every clone1 copy EAF 1
    eafs = {float(l.split("\t")[7][4:]) for l in pure}
    assert 0.0 in eafs and 1.0 in eafs


def test_truth_names_without_abundance_rows(built, workdir):
    """Four populations in name= and an abundance file without lines: the one sample draws from the first population alone,
    so only its segments are phased.  Its column carries the truth, the other columns are '.', and no CNV record of another
    population appears."""
    scn = helpers.build_scenario("se_tumor", os.path.join(workdir, "truth_noabund"))
    open(scn["kw"]["abundance"], "w").close()
    [body] = truth_round_trip(scn)
    assert body
    for l in body:
        cols = l.split("\t")[9:]
        assert cols[0] != "." and cols[1:] == [".", ".", "."], l
    assert sum("<CNV>" in l for l in body) == 1          # clone1's one 'c' record (200001-600000)


def test_truth_c_abi(built, workdir):
    """ssh_write_truth_vcf and its Python mirror Job.write_truth_vcf on a plan-only job (no device handle): SSC_ERR_STATE
    unless the sample is the one prepared last, SSC_ERR_INVALID for a sample the job does not have, SSC_ERR_SINK for a path
    that cannot be written, and the CLI's file otherwise."""
    import ctypes as C
    from simuscop_b200 import host_binding
    scn = helpers.build_scenario("se_tumor", os.path.join(workdir, "truth_abi"))
    _, out, r = run_plan_only(scn, "cli", truth=True)
    assert r.returncode == 0, r.stderr[-3000:]
    files = [helpers.read_file(os.path.join(out, s + ".truth.vcf")) for s in stems(scn)]
    cfg = os.path.join(scn["dir"], "cfg_abi.txt")
    synth.write_config(cfg, output=os.path.join(scn["dir"], "out_abi"), **scn["kw"])
    L = host_binding.lib()
    job = host_binding.Job(cfg, scn["seed"])
    try:
        path = os.path.join(scn["dir"], "abi.vcf")
        assert job.num_samples == 2
        assert L.ssh_write_truth_vcf(job.j, 0, path.encode()) == 3           # SSC_ERR_STATE: nothing prepared yet
        assert L.ssh_write_truth_vcf(job.j, 2, path.encode()) == 1           # SSC_ERR_INVALID
        assert not os.path.exists(path)
        pp, ep = C.c_int64(), C.c_int64()
        for s in range(2):
            assert L.ssh_prepare_sample(job.j, s, None, None, C.byref(pp), C.byref(ep)) == 0
            assert L.ssh_write_truth_vcf(job.j, s, os.path.join(scn["dir"], "no_such_dir", "x.vcf").encode()) == 5   # SSC_ERR_SINK
            job.write_truth_vcf(s, path)
            assert helpers.read_file(path) == files[s]
        assert L.ssh_write_truth_vcf(job.j, 0, path.encode()) == 3           # sample 1 was prepared since
        with pytest.raises(RuntimeError):
            job.write_truth_vcf(0, path)
    finally:
        job.close()


HAND_VARIATIONS = """\
c\ttest\tchr7\t1001\t2000\t3\t2
s\ttest\tchr7\t1500\t{b1500}\t{a1500}\thet
i\ttest\tchr7\t1200\tacg\thomo
d\ttest\tchr7\t1995\t10\thet
d\ttest\tchr7\t1\t2\thomo
s\ttest\tchr7\t3100\tA\tC\thomo
"""


def test_truth_hand_checked(built, workdir):
    """One 3 kb chromosome, ploidy 2, and a CN-3 segment (1001-2000).  The phasing draw gives haplotype index 0 two tandem
    copies and makes it the major set.  The variants:
      - het SNV at 1500: the first het SNV goes to the major set, so to both copies of index 0;
      - hom insertion ACG after 1200: on every copy;
      - het deletion of 1995-2004, which the first het deletion puts on index 0.  The reference erases 10 bases at the
        first copy's offset.  That takes 1995-2000 of copy 0 and 1001-1004 of copy 1, which is the copy junction.  The
        erase for copy 1 then starts at 1995 of copy 1 and stops at the string's end after 6 bases.  So copy 0 lacks
        1995-2000 (anchored on 1994), and copy 1 lacks 1001-1004 (anchored on 1000, in the previous segment) and 1995-2000;
      - SNP-file allele equal to the reference base at 2500: no record;
      - SNV at 3100, beyond the 3000-base chromosome: no record;
      - hom deletion of bases 1-2: anchored to the right, on base 3."""
    d = os.path.join(workdir, "truth_hand")
    os.makedirs(d, exist_ok=True)
    ref = "".join("ACGT"[(i * 7 + i // 5) % 4] for i in range(3000))
    synth.write_fasta(os.path.join(d, "ref.fa"), [("chr7 hand-made contig", np.frombuffer(ref.encode(), dtype=np.uint8))])
    alt1500 = {"A": "G", "C": "T", "G": "A", "T": "C"}[ref[1499]]
    with open(os.path.join(d, "v.txt"), "w") as f:
        f.write(HAND_VARIATIONS.format(b1500=ref[1499], a1500=alt1500))
    other = "A" if ref[2499] != "A" else "C"
    with open(os.path.join(d, "snp.txt"), "w") as f:
        f.write("rs1\tchr7\t2500\t%s/%s\t+\t%s\n" % (ref[2499], other, other))
    from simuscop_b200 import testdata
    data = testdata.materialize(os.path.join(workdir, "data"))
    scn = dict(dir=d, seed=5, name="hand", kw=dict(ref=os.path.join(d, "ref.fa"), profile=os.path.join(data, testdata.PROFILES["GAIIx"]),
                                                   layout="SE", coverage=1, insertSize=250, threads=1, verbose=0, name="test",
                                                   variation=os.path.join(d, "v.txt"), snp=os.path.join(d, "snp.txt")))
    [body] = truth_round_trip(scn)
    assert body == [
        "chr7\t1\t.\t%s\t%s\t.\tPASS\tEAF=1\tGT:HCN\t1|1:1,1" % (ref[0:3], ref[2]),
        "chr7\t1000\t.\t%s\t%s\t.\tPASS\tEAF=0.333333\tGT:HCN\t0|1|0:2,1" % (ref[999:1004], ref[999]),
        "chr7\t1001\t.\t%s\t<CNV>\t.\tPASS\tSVTYPE=CNV;END=2000\tCN:MCN:HCN\t3:2:2,1" % ref[1000],
        "chr7\t1200\t.\t%s\t%sACG\t.\tPASS\tEAF=1\tGT:HCN\t1|1|1:2,1" % (ref[1199], ref[1199]),
        "chr7\t1500\t.\t%s\t%s\t.\tPASS\tEAF=0.666667\tGT:HCN\t1|1|0:2,1" % (ref[1499], alt1500),
        "chr7\t1994\t.\t%s\t%s\t.\tPASS\tEAF=0.666667\tGT:HCN\t1|1|0:2,1" % (ref[1993:2000], ref[1993]),
    ]
    assert (ref[0:3], ref[999:1004], ref[1993:2000]) == ("ATG", "AATGC", "CAATGCA")


@pytest.mark.gpu
def test_truth_cli_on_gpu(built, workdir):
    """A pe_variants run with the truth on: the FASTQ files equal the run without it and the reference's (golden.json), the
    truth file equals the plan-only one, and sharding over SIMUSCOP_DEVICES writes the same file."""
    import torch
    scn = helpers.build_scenario("pe_variants", os.path.join(workdir, "truth_gpu"))
    gold = helpers.golden_entry("pe_variants")
    _, out_plan, r = run_plan_only(scn, "plan", truth=True)
    assert r.returncode == 0, r.stderr[-3000:]
    want = helpers.read_file(os.path.join(out_plan, "test.truth.vcf"))
    d = scn["dir"]
    fq = {}
    devs = "0,1" if torch.cuda.device_count() >= 2 else "0,0"
    for tag, extra in (("off", {}), ("on", {"SIMUSCOP_TRUTH_VCF": "1"}), ("sharded", {"SIMUSCOP_TRUTH_VCF": "1", "SIMUSCOP_DEVICES": devs})):
        out = os.path.join(d, "out_gpu_" + tag)
        cfg = os.path.join(d, "cfg_gpu_%s.txt" % tag)
        synth.write_config(cfg, output=out, **scn["kw"])
        env = dict(os.environ, SIMUSCOP_SEED=str(scn["seed"]), SIMUSCOP_BATCH_PAIRS="8192", **extra)
        if tag == "off":
            env.pop("SIMUSCOP_TRUTH_VCF", None)
        r = subprocess.run([SIMUREADS, cfg], env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        fq[tag] = [helpers.read_file(os.path.join(out, f)) for f in ("test_1.fq", "test_2.fq")]
        if tag == "off":
            assert sorted(os.listdir(out)) == ["test_1.fq", "test_2.fq"]
        else:
            assert helpers.read_file(os.path.join(out, "test.truth.vcf")) == want, tag
    assert fq["off"] == fq["on"] == fq["sharded"]
    s = gold["samples"][0]
    assert [hashlib.sha256(b).hexdigest() for b in fq["on"]] == [s["fq1_sha256"], s["fq2_sha256"]]
