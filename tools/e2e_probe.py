"""End-to-end MSM from pinned host buffers (development aid): python tools/e2e_probe.py [lgn]"""
import ctypes, os, random, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from python_bulletproofs_b200 import _native as nat
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
nat.init(0); lib = nat.load()
lib.bp_msm_set_host_finish(int(os.environ.get("BP_HOST_FINISH", "1")))
lgn = int(sys.argv[1]) if len(sys.argv) > 1 else 20
n = 1 << lgn
pts, sc = bench.synth_inputs(n, 7)
pp, ps = bench.pinned_copy(nat, pts), bench.pinned_copy(nat, sc)
out = ctypes.create_string_buffer(64)
ts = []
for it in range(12):
    a = time.perf_counter(); nat.check(lib.bp_msm_sharded_host(pp, ps, n, out)); ts.append((time.perf_counter() - a) * 1e3)
ts = sorted(ts[2:])
print("e2e 2^%d: median %.3f ms best %.3f ms -> %.1f Mpts/s (piece %s MiB)" % (lgn, ts[len(ts) // 2], ts[0], n / ts[len(ts) // 2] / 1e3,
      os.environ.get("BP_H2D_PIECE_MIB", "6")), flush=True)
