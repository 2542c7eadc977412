"""Every device form of the threshold compares and of the FP64 position against the C oracle, byte for byte, on the profiles of
draw_planting: thresholds planted exactly on (T = u) and one below (T = u - 1) the draws the reads make, for insert sizes,
indel lengths, substitution rows and quality rows (with 16-bit-key rows decided by the keys alone and by a key tie); rates
whose insertion and deletion tests pass at exactly one draw, none, or every draw (limits that wrap); and fragment positions
whose FP64 value rounds up across an integer.  A random draw meets its threshold with probability 2^-32, so the other suites
never test these inputs; test_draw_thresholds shows, without a GPU, that moving any site's thresholds by one changes the
bytes.  Every run asserts the instance it launched (ssc_stats gen_kernel / gen_nch / gen_qmode)."""
import pytest

import draw_planting as dp
from test_gpu_kernel_matrix import FAST, FP64, GENERIC_GLOBAL, GENERIC_SMEM, assert_same_fastq, check_path  # noqa: F401
from test_gpu_read_arrays import to_fastq

pytestmark = pytest.mark.gpu

GENERIC = (GENERIC_SMEM, 10, -1)
FP64_SEARCH = (FP64, 10, -1)

# case -> [(instance id, options, expected (gen_kernel, gen_nch, gen_qmode))]; "arrays": ssc_generate_reads
PLANTED = {
    "pe151": [("qp8", {}, (FAST, 5, 8)), ("qp2", {"fast_qmode": 2}, (FAST, 5, 2)), ("qp0", {"fast_qmode": 0}, (FAST, 5, 0)),
              ("generic", {"force_generic": 1}, GENERIC), ("fp64", {"fp64_search": 1}, FP64_SEARCH),
              ("arrays", {"arrays": 1}, (FAST, 5, 8))],
    "pe64": [("qp16", {}, (FAST, 2, 16)), ("qp2", {"fast_qmode": 2}, (FAST, 2, 2)), ("qp0", {"fast_qmode": 0}, (FAST, 2, 0)),
             ("generic", {"force_generic": 1}, GENERIC), ("arrays", {"arrays": 1}, (FAST, 2, 16))],
    "se97": [("qp8", {"fast_qmode": 8}, (FAST, 4, 8)), ("qp16", {"fast_qmode": 16}, (FAST, 4, 16)),
             ("generic", {"force_generic": 1}, GENERIC)],
    "k5": [("generic_global", {"force_generic": 1}, (GENERIC_GLOBAL, 10, -1))],
}
RATE_FAST = {"pe151": (FAST, 5, 8), "pe64": (FAST, 2, 16)}
RATE_MODES = [("fast", {}), ("no_splice", {"no_splice": 1}), ("generic", {"force_generic": 1}), ("fp64", {"fp64_search": 1})]
RATE_NAMES = ["ins_at", "ins_below", "del_at", "del_below", "del_at_ir", "del_below_ir", "ins_wrap", "ins_max", "del_wrap"]
POSITION = [("fast", {}, (FAST, 5, 8)), ("generic", {"force_generic": 1}, GENERIC), ("fp64", {"fp64_search": 1}, FP64_SEARCH),
            ("arrays", {"arrays": 1}, (FAST, 5, 8))]


def run(plan, options):
    """(FASTQ 1, FASTQ 2, stats) of the whole plan; with "arrays", the FASTQ the read arrays stand for."""
    from simuscop_b200 import cuda_binding
    options = dict(options)
    arrays = options.pop("arrays", 0)
    g = cuda_binding.Generator(0)
    try:
        for k, v in options.items():
            g.set_option(k, v)
        g.load_plan(plan, dp.SEED)
        if arrays:
            f1, f2 = to_fastq(g, g.generate_reads(0, g.planned))
        else:
            f1, f2 = g.generate()
        return f1, f2, g.stats()
    finally:
        g.close()


@pytest.fixture(scope="module")
def planted(built, workdir):
    cache = {}

    def get(name):
        if name not in cache:
            plan, _ = dp.plant_case(name, workdir)
            o1, o2, _ = dp.oracle(plan, trace=False)
            cache[name] = (plan, o1, o2)
        return cache[name]
    return get


@pytest.mark.parametrize("name,instance,options,want",
                         [pytest.param(n, i, o, w, id="%s-%s" % (n, i)) for n, runs in PLANTED.items() for i, o, w in runs])
def test_planted_thresholds(name, instance, options, want, planted, check_path):
    """Insert sizes, indel lengths, substitution and quality rows with thresholds on the reads' own draws: every quality
    mode of the fast kernel (QP 8's three-step search, QP 16's 16-bit keys and exact repeat, QP 2's ref == call rows, QP 0),
    the generic kernel with its tables in shared or global memory, the FP64 search and the array output."""
    plan, o1, o2 = planted(name)
    f1, f2, st = run(plan, options)
    assert_same_fastq((f1, f2), (o1, o2), "%s %s" % (name, instance))
    check_path(st, want)


@pytest.fixture(scope="module")
def rates(built, workdir):
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = {k: (plan, dp.oracle(plan, trace=False)[:2]) for k, (plan, _) in dp.rate_cases(name, workdir).items()}
        return cache[name]
    return get


@pytest.mark.parametrize("mode,options", [pytest.param(m, o, id=m) for m, o in RATE_MODES])
@pytest.mark.parametrize("case", RATE_NAMES)
@pytest.mark.parametrize("name", dp.RATE_PROFILES)
def test_rate_thresholds(name, case, mode, options, rates, check_path):
    """Insertion and deletion tests whose threshold is the smallest draw of the plan (exactly one event) or one below it
    (none), with insert_rate 0 and not; rates whose limit wraps (every read takes the slow path) or is the largest that does
    not; deletions clipped at the read end and reads that fall below 50 bases."""
    plan, (o1, o2) = rates(name)[case]
    f1, f2, st = run(plan, options)
    assert_same_fastq((f1, f2), (o1, o2), "%s %s %s" % (name, case, mode))
    check_path(st, {"generic": GENERIC, "fp64": FP64_SEARCH}.get(mode, RATE_FAST[name]))


@pytest.fixture(scope="module")
def positions(built, workdir):
    plan, cases = dp.position_case(dp.base_plan("pe151", workdir))
    o1, o2, _ = dp.oracle(plan, trace=False)
    return plan, cases, o1, o2


@pytest.mark.parametrize("mode,options,want", [pytest.param(m, o, w, id=m) for m, o, w in POSITION])
def test_position_rounding(mode, options, want, positions, check_path):
    """Fragment positions whose FP64 value (product, sum or both rounded; for both, a fused multiply-add would not round up)
    is one more than the exact quotient's floor, some with the contig end where only the exact position would leave a read:
    the position in the read name (and in the pos array) and the census's rejection of attempt 0 match the oracle on the fast
    kernel, the generic kernel and the FP64 search."""
    plan, cases, o1, o2 = positions
    f1, f2, st = run(plan, options)
    assert_same_fastq((f1, f2), (o1, o2), "positions %s" % mode)
    check_path(st, want)
