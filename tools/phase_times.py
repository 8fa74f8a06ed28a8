"""Where does one pass of the bench workload spend its time?  Wraps every Engine method with host timestamps and
CUDA events (development aid; run on the GPU box: PYTHONPATH=. python tools/phase_times.py [--precision tf32x3]).
--profile DIR: instead, one pass under torch.profiler (CUDA activities), its kernel and copy list written to
DIR/kernels.txt and the trace to DIR/trace.json (no wrappers: the profiler run is kept apart from the timeline)."""
import os as _os, sys as _sys
_sys.path.insert(0, _os.path.dirname(_os.path.dirname(_os.path.abspath(__file__))))
import argparse, json, time
import numpy as np, torch
import bench
from plspy_b200 import bootstrap_permutation as bp, class_functions as cf, resample
from plspy_b200.engine import Engine

ap = argparse.ArgumentParser()
ap.add_argument("--precision", default="fp64")
ap.add_argument("--voxels", type=int, default=bench.P_VOX)
ap.add_argument("--n", type=int, default=5000)
ap.add_argument("--profile", metavar="DIR", default=None)
a = ap.parse_args()

X = bench.make_data(p=a.voxels)
co = np.array([[n] * bench.C for n in bench.GROUPS])
_, X_mc = cf._mean_centre(X, co, 0)
U, s, V = cf._run_pls(X_mc)
Tvsc = cf._get_group_condition_means(X @ V, co)
np.random.seed(1)
ip = resample.permutation_indices("mct", a.n, co)[0]; ib = resample.bootstrap_indices("mct", a.n, co)[0]
dev = torch.device("cuda", 0)
Xd = torch.from_numpy(X).to(dev); Vd = torch.from_numpy(np.ascontiguousarray(V)).to(dev)
ipd = torch.from_numpy(ip.astype(np.int32)).to(dev); ibd = torch.from_numpy(ib.astype(np.int32)).to(dev)

log = []
def wrap(name, fn):
    def w(*args, **kw):
        t0 = time.perf_counter()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); out = fn(*args, **kw); e1.record()
        log.append((name, t0, time.perf_counter(), e0, e1))
        return out
    return w

def one():
    eng = Engine(Xd, device=dev, precision=a.precision)
    return bp.ResampleTest._create("mct", Xd, None, U, s.copy(), Vd, co, 0, preprocess=cf._mean_centre, nperm=a.n,
                                   nboot=a.n, Tvsc_orig=Tvsc, CI=0.95, perm_indices=ipd, boot_indices=ibd, engine=eng)


if a.profile:
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        one()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        one(); torch.cuda.synchronize()
    _os.makedirs(a.profile, exist_ok=True)
    prof.export_chrome_trace(_os.path.join(a.profile, "trace.json"))
    with open(_os.path.join(a.profile, "kernels.txt"), "w") as f:
        f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=60, max_name_column_width=70) + "\n")
        # device activity in start order, ms from the first one
        ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                    key=lambda e: e.time_range.start)
        t0 = ev[0].time_range.start if ev else 0
        for e in ev:
            f.write(f"{(e.time_range.start - t0) / 1e3:9.3f} {(e.time_range.end - e.time_range.start) / 1e3:8.3f}  "
                    f"{e.name[:110]}\n")
    print(open(_os.path.join(a.profile, "kernels.txt")).read())
    raise SystemExit(0)

for name in ("gram_of", "gram_stacked", "xv", "nspace", "pack_coef", "perm_count", "uhat", "boot_moments",
             "boot_count_gram", "boot_factor", "boot_factor_quad", "boot_finalize", "colstd", "to_host",
             "to_host_async", "to_device"):
    setattr(Engine, name, wrap(name, getattr(Engine, name)))
for _ in range(3):
    one()
torch.cuda.synchronize(); log.clear()
t0 = time.perf_counter(); one(); torch.cuda.synchronize(); t1 = time.perf_counter()
print(f"precision={a.precision} wall {1e3 * (t1 - t0):.2f} ms")
agg = {}
for name, h0, h1, e0, e1 in log:
    d = agg.setdefault(name, [0, 0.0, 0.0]); d[0] += 1; d[1] += 1e3 * (h1 - h0); d[2] += e0.elapsed_time(e1)
print(f"{'call':16s} {'n':>3s} {'host ms':>9s} {'gpu ms':>9s}")
for k, (n, h, g) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
    print(f"{k:16s} {n:3d} {h:9.3f} {g:9.3f}")
print("timeline (ms from start):")
for name, h0, h1, e0, e1 in log:
    print(f"  {1e3 * (h0 - t0):8.3f} -> {1e3 * (h1 - t0):8.3f}  {name}")
