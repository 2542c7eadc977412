"""Kernel-only probe: scale the read counts of a small plan of the C++ front end and time generate_device."""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers  # noqa: E402
from simuscop_b200 import cuda_binding, planfile  # noqa: E402

scale = int(sys.argv[1]) if len(sys.argv) > 1 else 256
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
prof = sys.argv[3] if len(sys.argv) > 3 else "XTen"
wd = "/tmp/qb"
helpers.SCENARIOS["qb"] = dict(lengths=[3000000], profile=prof, layout="PE", coverage=2, insertSize=300)
scn = helpers.build_scenario("qb", wd)
plan = planfile.read_plan(helpers.plan_dumps(scn, "qb")[0])
plan.bins["read_count"] *= scale
g = cuda_binding.Generator(0)
g.set_option("batch_pairs", int(os.environ.get("QB_BATCH", 1 << 21)))
if os.environ.get("QB_GZIP"):
    g.set_option("gzip", 1)
for kv in filter(None, os.environ.get("QB_OPTS", "").split(",")):          # e.g. QB_OPTS=concurrent_move=0
    g.set_option(kv.split("=")[0], int(kv.split("=")[1]))
t = time.time()
g.load_plan(plan, 7)
print("load_plan %.2fs planned=%d emitted=%d" % (time.time() - t, g.planned, g.emitted))
for r in range(reps):
    g.reset_stats()
    res = g.generate_device()
    st = g.stats()
    tot = res["bytes1"] + res["bytes2"] + st["hap_bytes"]
    print("rep %d: %.3f ms  %.1f Gbases/s  fastq %.1f GB/s  algorithmic %.1f GB/s (%.1f%% of 6554)  launches %d  gen %.3f ms/batch  pass2 %.3f ms/batch" % (
        r, res["device_ms"], res["bases"] / res["device_ms"] / 1e6, (res["bytes1"] + res["bytes2"]) / res["device_ms"] / 1e6,
        tot / res["device_ms"] / 1e6, 100 * tot / res["device_ms"] / 1e6 / 6554.2, st["launches"],
        st["gen_kernel_ms"] / max(1, st["timed_batches"]), st["compact_kernel_ms"] / max(1, st["timed_batches"])))
