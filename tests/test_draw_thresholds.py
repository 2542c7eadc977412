"""The profiles of draw_planting, checked without a GPU: the planted thresholds are what the host tables and the FP64 randIndx
make of them, the final plans still make the planted draws (per site, per threshold slot, per 16-bit-key kind), moving the
planted thresholds of a site by one changes the FASTQ (so an off-by-one compare of that site on the device could not pass
test_gpu_draw_thresholds), the rate cases make exactly the one event they are built for, and the position cases round.

Also pins the oracle's draw trace (it changes no byte; its words are the Philox words of the draw addresses) and the numpy
Philox the planting uses."""
import numpy as np
import pytest

import draw_planting as dp

CASES = ("pe151", "pe64", "se97", "k5")

# what the builder achieves, rounded down: planted thresholds whose draw the final plan makes, by (site, kind) ...
COVERAGE_FLOOR = {
    "pe151": {("isize", "at"): 20, ("isize", "past"): 19, ("inslen", "at"): 5, ("inslen", "past"): 6, ("dellen", "at"): 10,
              ("dellen", "past"): 9, ("sub", "at"): 8000, ("sub", "past"): 8000, ("qual", "at"): 2350, ("qual", "past"): 2350},
    "pe64": {("isize", "at"): 20, ("isize", "past"): 19, ("inslen", "at"): 5, ("inslen", "past"): 6, ("dellen", "at"): 10,
             ("dellen", "past"): 9, ("sub", "at"): 5500, ("sub", "past"): 5500, ("qual", "at"): 5400, ("qual", "past"): 5400,
             ("qual", "key_below"): 2700, ("qual", "key_above"): 2700, ("qual", "key_tie"): 2700},
    "se97": {("inslen", "at"): 5, ("inslen", "past"): 6, ("dellen", "at"): 10, ("dellen", "past"): 9, ("sub", "at"): 4350,
             ("sub", "past"): 4350, ("qual", "at"): 1900, ("qual", "past"): 1900},
    "k5": {("isize", "at"): 20, ("isize", "past"): 19, ("inslen", "at"): 5, ("inslen", "past"): 6, ("dellen", "at"): 10,
           ("dellen", "past"): 9, ("sub", "at"): 9400, ("sub", "past"): 9400, ("qual", "at"): 140, ("qual", "past"): 140},
}
# ... and FASTQ records that change when a site's planted thresholds move by one
SENSITIVITY_FLOOR = {
    "pe151": {"isize": 39, "inslen": 11, "dellen": 18, "sub": 1900, "qual": 1700},
    "pe64": {"isize": 39, "inslen": 11, "dellen": 15, "sub": 7800, "qual": 7800},
    "se97": {"inslen": 11, "dellen": 18, "sub": 3450, "qual": 2450},
    "k5": {"isize": 39, "inslen": 11, "dellen": 17, "sub": 2750, "qual": 270},
}
SLOTS = {"isize": 39, "inslen": 11, "dellen": 19, "sub": 3}


@pytest.fixture(scope="module")
def planted(built, workdir):
    cache = {}

    def get(name):
        if name not in cache:
            plan, pl = dp.plant_case(name, workdir)
            cache[name] = (plan, pl, dp.oracle(plan))
        return cache[name]
    return get


def test_philox_known_answer_and_trace_words(built, workdir):
    """The numpy Philox4x32-10 gives the Random123 known answer and the oracle's words; every word of the oracle's draw
    trace is the Philox word of its address."""
    from oracle import binding as oracle_binding
    assert [int(x) for x in dp.philox(0, 0, 0, 0, 0, 0)] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert [int(x) for x in oracle_binding.philox([0] * 4, [0, 0])] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    rng = np.random.default_rng(1)
    for _ in range(50):
        c, k = rng.integers(0, 1 << 32, 4, dtype=np.uint64), rng.integers(0, 1 << 32, 2, dtype=np.uint64)
        assert [int(x) for x in dp.philox(*c, int(k[0]), int(k[1]))] == [int(x) for x in oracle_binding.philox(c, k)]
    plan = dp.base_plan("pe151", workdir, small=True)
    _, _, info = dp.oracle(plan)
    f, s, b = info["frag"], info["scan"], info["base"]
    w = dp.block(dp.SEED, f["pair"].astype(np.uint64), 0, dp.STREAM_FRAG, 0, f["attempt"])
    assert (w[0] == f["x0"]).all() and (w[1] == f["x1"]).all()
    w = dp.block(dp.SEED, s["pair"].astype(np.uint64), s["mate"], dp.STREAM_CYCLE, 0, s["j"])
    assert (w[0] == s["x0"]).all() and (w[1] == s["x1"]).all()
    w = dp.block(dp.SEED, b["pair"].astype(np.uint64), b["mate"], dp.STREAM_CYCLE, 0, b["j"])
    assert (w[2] == b["u2"]).all() and (w[3] == b["u3"]).all()
    ev = s[s["kind"] > 0]
    w = dp.block(dp.SEED, ev["pair"].astype(np.uint64), ev["mate"], dp.STREAM_LEN, 0, ev["j"])
    assert len(ev) and (np.where(ev["kind"] == 1, w[0], w[1]) == ev["lenword"]).all()


def test_draw_trace_changes_no_byte(planted):
    """The same FASTQ with the draw trace on and off; one trace row per attempt, scanned position and output base."""
    plan, _, (f1, f2, info) = planted("pe151")
    g1, g2, plain = dp.oracle(plan, trace=False)
    assert (g1, g2) == (f1, f2) and plain["bases"] == info["bases"] == len(info["base"])
    assert info["frag"]["accepted"].sum() == info["emitted"]
    reads = info["frag"]["accepted"].sum() * (2 if plan.paired else 1)
    assert len(info["scan"]) == reads * plan.hdr["read_length"] - _skipped(info["scan"], plan.hdr["read_length"])


def _skipped(scan, RL):
    """Positions the scan steps over: the tail of each deletion (clipped at the read end)."""
    d = scan[(scan["kind"] == 2) & (scan["k"] > 0)]
    return int(np.minimum(d["k"], RL - d["j"]).sum() - len(d))


def _row_cdf(plan, p):
    if p.site == "isize":
        return plan.tables["isize_cdf"]
    if p.site in ("inslen", "dellen"):
        return plan.tables["ins_cdf" if p.site == "inslen" else "del_cdf"]
    B, R = plan.hdr["bins"], plan.hdr["n_kmer_rows"]
    if p.site == "sub":
        tab, row = divmod(p.row, R * B)
        return plan.tables["subs_cdf%d" % (tab + 1)].reshape(-1, 4)[row]
    return plan.tables["quality_cdf"].reshape(-1, plan.hdr["n_qual"])[p.row]


@pytest.mark.parametrize("name", CASES)
def test_construction(name, planted):
    """Every planted threshold: the host tables (ssc_table_lookup_host / ssc_sub_lookup_host) and the FP64 randIndx agree at
    u - 1, u and u + 1, and the decision changes exactly between T and T + 1 (at: u takes the lower symbol, one past: the
    higher one; the 16-bit-key kinds are on the side of T they were built for)."""
    from oracle import binding as oracle_binding
    from simuscop_b200 import cuda_binding
    L, O = cuda_binding.lib(), oracle_binding.lib()
    plan, pl, _ = planted(name)
    for p in pl:
        cdf = np.ascontiguousarray(_row_cdf(plan, p))
        n = cdf.size

        def host(u):
            return L.ssc_sub_lookup_host(cdf.ctypes.data, u) if p.site == "sub" else L.ssc_table_lookup_host(cdf.ctypes.data, n, u)
        for u in (p.u - 1, p.u, p.u + 1, p.T, p.T + 1):
            assert host(u) == O.ssco_rand_indx(cdf.ctypes.data, n, u), (p, u)
        assert O.ssco_rand_indx(cdf.ctypes.data, n, p.T) < O.ssco_rand_indx(cdf.ctypes.data, n, p.T + 1), p
        assert (p.u <= p.T) == (p.kind in ("at", "key_above", "key_tie")), p
        if p.kind.startswith("key"):
            assert {"key_below": (p.u >> 16) - 1, "key_above": (p.u >> 16) + 1, "key_tie": p.u >> 16}[p.kind] == p.T >> 16, p


@pytest.mark.parametrize("name", CASES)
def test_coverage(name, planted):
    """The final plan makes at least COVERAGE_FLOOR planted draws per site and kind; every threshold slot of the substitution
    and quality searches (0..2, 0..live - 2) has a draw at and one past its threshold in some row, and every slot of the
    one-row tables (insert size 0..38, lengths 0..10 / 0..18) a draw at or one past it."""
    plan, pl, (_, _, info) = planted(name)
    total, per_slot = dp.coverage(plan, pl, info)
    short = {k: (total.get(k, 0), v) for k, v in COVERAGE_FLOOR[name].items() if total.get(k, 0) < v}
    assert not short, short
    slots = dict(SLOTS, qual=dp.PROFILES[name]["live"] - 1)
    for site in {p.site for p in pl}:
        for slot in range(slots[site]):
            got = [kind for kind in ("at", "past") if per_slot.get((site, slot, kind), 0) > 0]
            assert got == ["at", "past"] if site in ("sub", "qual") else got, (site, slot, got)


@pytest.mark.parametrize("name", CASES)
def test_sensitivity(name, planted):
    """Moving one site's planted thresholds by one (what a < for <= or a lost + 1 amounts to) changes at least
    SENSITIVITY_FLOOR FASTQ records of the oracle: the byte comparison on the GPU sees an off-by-one of any site."""
    plan, pl, (f1, f2, _) = planted(name)
    got = {}
    for site in SENSITIVITY_FLOOR[name]:
        g1, g2, _ = dp.oracle(dp.move_by_one(plan, pl, site), trace=False)
        got[site] = dp.differing_records((f1, f2), (g1, g2))
    short = {s: (got[s], v) for s, v in SENSITIVITY_FLOOR[name].items() if got[s] < v}
    assert not short, short


@pytest.mark.parametrize("name", dp.RATE_PROFILES)
def test_rate_cases(name, built, workdir):
    """insert_rate = u*/2^32 makes exactly the one insertion at the smallest x0, (u* - 1)/2^32 none; the deletion rates whose
    FP64 quotient lies just above / below the smallest x1 make exactly one deletion / none, with insert_rate 0 and not; rates
    of 1 (limits that wrap) and (2^32 - 2)/2^32 pass the test at every position, with lengths that clip at the read end and
    reads that fall below 50 bases."""
    RL = dp.PROFILES[name]["kw"]["read_length"]
    for tag, (plan, want) in dp.rate_cases(name, workdir).items():
        _, _, info = dp.oracle(plan)
        s = info["scan"]
        ev = s[(s["kind"] > 0) & (s["k"] > 0)]
        if want is None:
            assert len(ev) == 0, (tag, ev[:3])
        elif want == "edge":
            kind = 2 if tag == "del_wrap" else 1
            assert (s["kind"] == kind).all(), tag
            assert len(ev) > 20, tag
            if kind == 2:
                assert (ev["k"] > RL - ev["j"]).any(), "no deletion clipped at the read end"
                assert (ev["k"] == RL - 49).any() and (ev["k"] == 3).any()
                reset = info["base"][info["base"]["j"] == 0]
                assert (reset["m"] == RL).any() and (reset["m"] < RL).any()
        else:
            kind = 1 if want[0] == "ins" else 2
            assert len(ev) == 1 and (int(ev[0]["kind"]), int(ev[0]["pair"]), int(ev[0]["mate"]), int(ev[0]["j"])) == \
                (kind,) + want[1:], (tag, ev)
            if kind == 1:
                assert plan.hdr["insert_rate"] * dp.TWO32 == int(ev[0]["x0"])
            else:
                q = np.float64(plan.hdr["del_rate"]) / (1.0 - np.float64(plan.hdr["insert_rate"]))
                assert int(ev[0]["x1"]) / dp.TWO32 < q <= (int(ev[0]["x1"]) + 1) / dp.TWO32


def test_position_cases(built, workdir):
    """Every planted pair's FP64 position (numpy float64, the reference's operation order) is one more than the exact
    floor(spos + span * u / 2^32); the oracle draws that position, and rejects attempt 0 where the contig end leaves the FP64
    position RL - 1 bases.  Every rounding occurs: the product (span >= 2^22), the sum (spos >= 2^24), and both, where one
    fused multiply-add would give the exact floor."""
    plan, cases = dp.position_case(dp.base_plan("pe151", workdir))
    RL = plan.hdr["read_length"]
    kinds = [c[4] for c in cases]
    assert kinds.count("product") >= 150 and kinds.count("sum") >= 30 and kinds.count("double") >= 10
    assert sum(c[5] for c in cases) >= 60
    _, _, info = dp.oracle(plan)
    f = info["frag"]
    first = {int(p): (int(pos), int(acc), int(ln)) for p, a, pos, acc, ln in zip(f["pair"], f["attempt"], f["pos"], f["accepted"],
                                                                                f["len"]) if a == 0}
    for pid, spos, span, u, kind, end_case in cases:
        exact = (spos * (1 << 32) + span * u) >> 32
        fp = int(np.float64(spos) + np.float64(span) * (np.float64(u) / dp.TWO32))
        assert fp == exact + 1, (pid, spos, span, u)
        fused = int((spos * (1 << 32) + span * u) / (1 << 32))      # one rounding of the exact value
        assert fused == (exact if kind == "double" else fp), (pid, kind)
        if kind == "product":
            assert (1 << 22) <= span < (1 << 25)
        elif kind == "double":
            assert (1 << 21) <= span < (1 << 22) and (1 << 24) <= spos < (1 << 25)
        else:
            assert span < (1 << 21) and (1 << 24) <= spos < (1 << 25)
        pos, acc, ln = first[pid]
        assert pos == fp and acc == (not end_case), (pid, pos, acc)
        if end_case:
            assert ln == RL - 1
