"""CPU arm of the benchmark (ORACLE — test / measurement infrastructure, not product code).

    python oracle/cpu_arm.py --steps K --warmup W [--config C4] [--per-step 2097152] [--json]

Times oracle/ref_eval.c (the plain-C restatement of the path, see its header for the reference lines it
follows) on the host cores of this box, and prints one JSON object.  bench.py runs this file as a
SUBPROCESS for both its `cpu_baseline` leg and `--impl reference`, so that the two legs are the same
measurement and neither inherits a thread count from an imported torch (round-1 VERDICT, weak §4:
omp_get_max_threads() changed once torch was loaded, and 200 000 candidates over 128 threads with a static
schedule made the rate move 5x between boxes).

What makes the number reproducible:
  * thread count fixed ONCE = physical cores this process may use (unique (package, core) pairs of the
    CPUs in the affinity mask, capped by the cgroup CPU quota), printed in the result;
  * OMP_PROC_BIND=close, OMP_PLACES=cores, OMP_DYNAMIC=false set before the library is loaded;
  * the C file is compiled on THIS host with -O3 -march=native (-ffp-contract=off kept: results stay
    bit-identical to the portable -O2 build the parity tests use) into a temporary directory, so that the
    benchmark writes nothing into the repository tree (which may be read-only);
  * a step is >= 2 M candidate evaluations (a 262 144-candidate sample evaluated repeatedly; the table and
    the sample exceed L2 per core, each candidate is an independent 256-step dependent chain);
  * OpenMP schedule(dynamic) over blocks of candidates; value = median over the timed steps.
"""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import tempfile
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def physical_cores():
    """(threads to use, description).  Physical cores among the CPUs this process may run on, capped by
    the cgroup quota (a container with a 32-CPU quota on a 128-thread host must not spawn 128 threads)."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
    except AttributeError:
        allowed = list(range(os.cpu_count() or 1))
    cores = set()
    for c in allowed:
        base = "/sys/devices/system/cpu/cpu%d/topology/" % c
        try:
            with open(base + "physical_package_id") as f:
                pkg = f.read().strip()
            with open(base + "core_id") as f:
                core = f.read().strip()
            cores.add((pkg, core))
        except OSError:
            cores.add(("?", str(c)))
    n = max(1, len(cores))
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                txt = f.read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                        quota = q / float(f.read().strip())
            break
        except (OSError, ValueError, IndexError):
            continue
    desc = "%d physical cores of %d allowed logical CPUs" % (n, len(allowed))
    if quota is not None and quota < n:
        n = max(1, int(math.floor(quota)))
        desc += ", capped by cgroup quota %.1f" % quota
    return n, desc


def native_build(out_dir):
    """gcc -O3 -march=native of oracle/ref_eval.c for this host -> out_dir/libref_eval_native.so"""
    src = os.path.join(HERE, "ref_eval.c")
    so = os.path.join(out_dir, "libref_eval_native.so")
    flags = ["-O3", "-march=native", "-fopenmp", "-shared", "-fPIC", "-ffp-contract=off"]
    try:
        subprocess.check_call(["gcc"] + flags + [src, "-o", so, "-lm"])
    except (OSError, subprocess.CalledProcessError):
        # no compiler on this host: fall back to the portable oracle/libref_eval.so the package build made
        sys.path.insert(0, ROOT)
        from oracle import c_oracle
        return c_oracle.build(), "gcc -O2 (portable build; native compile failed)"
    return so, "gcc " + " ".join(flags[:2])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--config", default="C4")
    ap.add_argument("--per-step", type=int, default=2 * 1024 * 1024)
    ap.add_argument("--sample", type=int, default=262144)
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--max-seconds", type=float, default=150.0, help="stop adding timed steps after this long")
    args = ap.parse_args()

    threads, how = physical_cores()
    if args.threads > 0:
        threads, how = args.threads, "forced by --threads"
    os.environ["OMP_NUM_THREADS"] = str(threads)
    os.environ["OMP_PROC_BIND"] = "close"
    os.environ["OMP_PLACES"] = "cores"
    os.environ["OMP_DYNAMIC"] = "false"
    os.environ.setdefault("OMP_WAIT_POLICY", "active")

    with tempfile.TemporaryDirectory(prefix="saturn_b200_cpu_arm_") as tmp:
        so, build = native_build(tmp)
        lib = ctypes.CDLL(so)                         # stays mapped after the directory is removed
    fn = lib.ref_eval_f32
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                   ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                   ctypes.c_void_p, ctypes.c_int]

    sys.path.insert(0, ROOT)
    import numpy as np
    from oracle import ref_eval as R
    from saturn_b200.synth import CONFIGS
    J, S, G, _seed = CONFIGS[args.config]
    T, valid = R.synth_table(J, S, G, seed=0)
    tab = np.ascontiguousarray(R.canon_table(T, range(1, G + 1)), dtype=np.float32)
    nsample = min(args.sample, args.per_step)
    opt, prio = R.synth_candidates(J, nsample, valid, seed=1)
    opt = np.ascontiguousarray(opt, dtype=np.uint8)
    prio = np.ascontiguousarray(prio)
    mk = np.empty(nsample, dtype=np.float32)
    reps = max(1, -(-args.per_step // nsample))
    per_step = reps * nsample

    def step():
        for _ in range(reps):
            rc = fn(tab.ctypes.data, J, S, opt.ctypes.data, prio.ctypes.data, prio.dtype.itemsize, nsample, 1, 8, 1,
                    mk.ctypes.data, None, None, threads)
            if rc != 0:
                raise RuntimeError("ref_eval_f32 rc=%d" % rc)

    t_begin = time.perf_counter()
    for _ in range(max(0, args.warmup)):
        step()
    times = []
    for _ in range(max(1, args.steps)):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_begin > args.max_seconds and len(times) >= 3:
            break
    times_sorted = sorted(times)
    med = times_sorted[len(times_sorted) // 2]
    total = sum(times)
    out = {
        "value": per_step / med, "unit": "candidates/s", "cores": threads, "cores_how": how, "kind": "port",
        "candidates_per_step": per_step, "steps_timed": len(times), "ms_per_step_median": med * 1e3,
        "ms_per_step_min": times_sorted[0] * 1e3, "ms_per_step_max": times_sorted[-1] * 1e3,
        "mean_value": per_step * len(times) / total, "seconds_timed": total, "build": build,
        "checksum": float(mk[:1024].astype(np.float64).sum()),
        "sample": "%d candidate evaluations per step (a %d-candidate sample of %s: J=%d,S=%d,G=%d, %d passes), "
                  "oracle/ref_eval.c fp32 integer starts, %s, OpenMP schedule(dynamic) on %d threads bound to cores "
                  "(%s), median of %d steps" % (per_step, nsample, args.config, J, S, G, reps, build, threads, how,
                                                len(times)),
    }
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
