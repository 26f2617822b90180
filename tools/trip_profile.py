"""Where one trip of the merged FP64 BULK launch (the fold body, SpecCassieFeetPelvisFold) spends its cycles: the library
rebuilt with IKB_TRIP_PROFILE=1 (dls_spec.cuh, TripClock) adds up clock64() deltas per segment of a trip and per warp
role, and this script prints cycles per trip for each.  Two builds are compared: `direct` (IKB_PREFETCH=0: every slot
refills from global memory at the end of its trip) and `staged` (the library's default: a converged slot's next problem is
staged one trip ahead).

    python tools/trip_profile.py --build        # compile both builds under build/trip_profile/ (no GPU needed)
    python tools/trip_profile.py [--steps 48]   # run the bench-shaped queue (65 536 per batch, merge 8, depth 24) on each

The instrumented object is compiled from this checkout's sources and linked with build/obj (run `make` first); the
library itself is never built with the counters.  The counters cost registers: the instrumented merged fold body spills
about 240 B per thread where the library's spills 8 B (--build prints it), so the segment cycles describe a slower
register allocation than the production kernel's -- read them as shares of a trip, not as its absolute length."""
import argparse
import ctypes
import glob
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "build", "trip_profile")
VARIANTS = {"direct": ["-DIKB_PREFETCH=0"], "staged": []}
SEGS = ["top bar.red", "tmem fetch q", "evaluate", "phase 1 + bar 1", "stop test", "phase 2/3", "barrier 2", "step",
        "results", "refill", "tmem park"]


def build():
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    flags = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
             "--expt-relaxed-constexpr", "-DIKB_TRIP_PROFILE=1"]
    objs = [o for o in glob.glob(os.path.join(ROOT, "build", "obj", "*.o")) if "spec_cassie_feet_pelvis" not in o]
    for name, extra in VARIANTS.items():
        tree = os.path.join(OUT, name)
        shutil.rmtree(tree, ignore_errors=True)
        shutil.copytree(os.path.join(ROOT, "ik_b200"), os.path.join(tree, "ik_b200"),
                        ignore=shutil.ignore_patterns("csrc", "libikb200.so", "__pycache__"))
        obj = os.path.join(tree, "spec_cassie_feet_pelvis.o")
        log = subprocess.run([nvcc] + flags + extra + ["-Xptxas", "-v", "-c", os.path.join(ROOT, "ik_b200", "csrc", "spec_cassie_feet_pelvis.cu"),
                              "-o", obj], check=True, capture_output=True, text=True).stderr.splitlines()
        # the counters cost registers: say what the instrumented merged fold body spills (the library's build: profiles/)
        for i, ln in enumerate(log):
            if "Function properties" in ln and "SpecCassieFeetPelvisFoldEdLi6ELi1ELb1E" in ln:
                print("%s: instrumented merged fold body:%s" % (name, log[i + 1].strip().split("stack frame,")[-1]))
        subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o",
                               os.path.join(tree, "ik_b200", "libikb200.so"), obj] + objs)
        print("built", tree)


def run_one(name, steps, batch):
    sys.path.insert(0, os.path.join(OUT, name))
    sys.path.insert(1, ROOT)
    import numpy as np
    import torch
    import ik_b200 as ik
    from ik_b200 import _capi
    from ik_b200 import workloads as W
    assert ik.__file__.startswith(OUT), ik.__file__
    assert torch.cuda.is_available(), "needs a GPU"
    read = _capi.lib.ikb_trip_profile
    read.argtypes = [ctypes.POINTER(ctypes.c_ulonglong), ctypes.c_int]
    dev = torch.device("cuda:0")
    pb = W.cassie_feet_pelvis_problem()
    pb.finalize(0)
    m = pb.model()
    sets = []
    for s in range(4):   # the inputs of tools/bulk_kernel_profile.py
        qstar = W.sample_configurations(m, batch, seed=100 + s)
        names = W.task_frames(pb)
        poses_t = ik.fk_batch(pb, torch.tensor(qstar.T.copy(), device=dev), names)
        poses = {n: poses_t[12 * i:12 * i + 12].T.cpu().numpy() for i, n in enumerate(names)}
        tg = W.targets_from_frame_poses(pb, poses)
        q0 = np.tile(W.standing_configuration(m, W.CASSIE_STANDING), (batch, 1))
        sets.append((torch.tensor(q0.T.copy(), device=dev), torch.tensor(tg.T.copy(), device=dev)))
    prm = ik.dls_parameters()
    queue = ik.SolveQueue(pb, 24, 8, 0)

    def run(n):
        for k in range(n):
            queue.submit(*sets[k % len(sets)], prm)
        queue.drain()
        torch.cuda.synchronize()

    run(16)
    n = 2 * (len(SEGS) + 1)
    buf = (ctypes.c_ulonglong * (4 * (len(SEGS) + 1)))()
    assert read(None, n) == 0
    run(steps)
    assert read(buf, n) == 0
    c = np.array(buf[:n], dtype=np.float64).reshape(2, len(SEGS) + 1)
    print("[%s] %s, %d steps of %d problems: cycles per trip (clock64, summed over warps / trips)" %
          (name, torch.cuda.get_device_name(0), steps, batch))
    print("%-18s %10s %10s" % ("segment", "role 0", "role 1"))
    for k, s in enumerate(SEGS):
        print("%-18s %10.0f %10.0f" % (s, c[0, k] / c[0, -1], c[1, k] / c[1, -1]))
    print("%-18s %10.0f %10.0f" % ("trip", c[0, :-1].sum() / c[0, -1], c[1, :-1].sum() / c[1, -1]))
    print("%-18s %10d %10d" % ("warp-trips", c[0, -1], c[1, -1]))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--build", action="store_true")
    ap.add_argument("--steps", type=int, default=48)
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--variant", choices=sorted(VARIANTS))
    args = ap.parse_args()
    if args.build:
        build()
    elif args.variant:
        run_one(args.variant, args.steps, args.batch)
    else:
        for name in VARIANTS:   # one process per build: both load a library named ik_b200
            subprocess.check_call([sys.executable, os.path.abspath(__file__), "--variant", name, "--steps", str(args.steps),
                                   "--batch", str(args.batch)])
