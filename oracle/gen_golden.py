"""Generate golden fixtures by running the UNMODIFIED reference solver.

ORACLE INFRASTRUCTURE.  Runs only in the build container (needs /root/reference);
the GPU box never executes this — it consumes the committed JSON under
tests/golden/.

    python oracle/gen_golden.py            # writes tests/golden/milp_cases.json

What it does: puts oracle/shims (pulp -> scipy HiGHS, ray -> 1 node x 8 GPUs)
and /root/reference on sys.path, imports the reference's `saturn.solver`, and
calls `solve()` + `convert_into_comprehensible()` on small duck-typed tasks
built from the reference's own `Strategy` class.  Two variants per case:

  as_shipped : milp.py byte-for-byte (M = 1e10, milp.py:163).  Under HiGHS'
               1e-6 integrality tolerance this big-M leaks (SURVEY §8c O1) and
               may return overlapping schedules — recorded, with the overlap
               count, as documentation of the hazard.
  tight_m    : the same source with the single literal `M = 1e10` replaced at
               load time by a sound horizon (sum of ceil(max runtime) + 1); the
               file on disk is untouched.  This is the MILP the oracle is
               pinned against.
"""
import importlib
import json
import math
import os
import random
import sys
import time
import types

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"


def _load_reference():
    for m in [m for m in sys.modules if m == "saturn" or m.startswith("saturn.")]:
        del sys.modules[m]
    sys.path[:] = [p for p in sys.path if os.path.abspath(p or ".") != os.path.dirname(HERE)]
    sys.path.insert(0, REF)
    sys.path.insert(0, os.path.join(HERE, "shims"))
    import saturn.solver.milp as milp  # noqa: the reference, unmodified
    assert milp.__file__.startswith(REF), milp.__file__
    src = open(milp.__file__).read()
    assert src.count("M = 1e10") == 1
    tight_src = src.replace(
        "M = 1e10",
        "M = float(__import__('os').environ.get('ORACLE_BIG_M_FACTOR', '1')) * "
        "float(sum(__import__('math').ceil(max(rt for (_g, rt) in tup)) for tup in gpu_time_tuples) + 1)")
    tight = types.ModuleType("saturn_solver_milp_tightM")
    tight.__file__ = milp.__file__ + " [M substituted at load time]"
    exec(compile(tight_src, tight.__file__, "exec"), tight.__dict__)
    from saturn.core.representations import Strategy
    import pulp
    return milp, tight, Strategy, pulp


class DuckTask:
    """What solve()/convert_into_comprehensible() touch on a Task (milp.py:77-81, 481-486)."""

    def __init__(self, name, strategies):
        self.name = name
        self.strategies = strategies
        self.selected_strategy = None

    def select_strategy(self, s):
        self.selected_strategy = s


def probe_tuples(J, options, seed):
    """SURVEY §8c known-answer generator: base ~ U(500,4000), T = base / g**0.8."""
    random.seed(seed)
    out = []
    for _ in range(J):
        base = random.uniform(500, 4000)
        out.append([(g, base / g ** 0.8) for g in options])
    return out


def hetero_tuples(J, seed):
    """Per-task option lists of different lengths/orders (dict-insertion order matters)."""
    rnd = random.Random(seed)
    out = []
    for _ in range(J):
        base = rnd.uniform(200, 2000)
        opts = rnd.sample([1, 2, 3, 4, 6, 8], rnd.randint(1, 3))
        out.append([(g, base * rnd.uniform(1.0, 1.3) / g ** rnd.uniform(0.5, 0.95)) for g in opts])
    return out


def run_case(mod, Strategy, pulp, name, tuples, timeout):
    tasks = []
    for t, tup in enumerate(tuples):
        strategies = {}
        for (g, rt) in tup:
            strategies[g] = Strategy("exec%d" % g, g, {}, rt)
        tasks.append(DuckTask("t%d" % t, strategies))
    t0 = time.time()
    sta, tga, bss, bna, boa, saved = mod.solve(tasks, None, gurobi=False, threads=1, interval=1000,
                                               timeout=timeout)
    wall = time.time() - t0
    info = dict(pulp.LpProblem.last_info)
    rec = {"name": name, "gpu_time_tuples": [[list(x) for x in tup] for tup in tuples],
           "solver_wall_s": wall, "highs": info, "returned_makespan": saved}
    if sta is None or any(v is None for n in sta for g in n for v in g):
        rec["incumbent"] = False
        return rec
    rec["incumbent"] = True
    rec.update({"sta": sta, "tga": tga, "bss": bss, "bna": bna, "boa": boa})
    npt, tdd, start = mod.convert_into_comprehensible(tasks, bss, boa, tga, bna, sta)
    idx = {t: i for i, t in enumerate(tasks)}
    rec["decoded"] = {
        "node_per_task": [int(npt[t]) for t in tasks],
        "deps": [sorted(idx[d] for d in tdd[t]) for t in tasks],
        "start": [float(s) for s in start],
        "selected_gpus": [int(t.selected_strategy.gpu_apportionment) for t in tasks],
    }
    rec["makespan"] = max(float(s) + t.selected_strategy.runtime for s, t in zip(start, tasks))
    return rec


def main_nodes(nodes):
    """Multi-node fixtures: the reference with ray.nodes() reporting `nodes` nodes (milp.py:58)."""
    os.environ["ORACLE_RAY_NODES"] = str(nodes)
    milp, tight, Strategy, pulp = _load_reference()
    sys.path.insert(0, os.path.dirname(HERE))
    from oracle import ref_eval as R
    cases = [
        ("N2_K1_J3_g8_seed1", probe_tuples(3, [8], 1), 120),
        ("N2_J4_g48_seed5", probe_tuples(4, [4, 8], 5), 240),
        ("N2_J3_g1248_seed0", probe_tuples(3, [1, 2, 4, 8], 0), 240),
        ("N2_J5_g8_seed4", probe_tuples(5, [8], 4), 240),
    ]
    out = {"generator": "oracle/gen_golden.py --nodes %d" % nodes, "reference_commit": "b65e3d2", "nodes": nodes,
           "scipy": __import__("scipy").__version__, "cases": []}
    for name, tuples, timeout in cases:
        rec = run_case(tight, Strategy, pulp, name, tuples, timeout)
        rec["variant"] = "tight_m"
        rec["proven_optimal"] = bool(rec["highs"].get("status") == 0)
        if rec["incumbent"]:
            plan = R.plan_from_arrays(tuples, rec["sta"], rec["tga"], rec["bss"], rec["bna"])
            ok, ov, mk = R.check_plan([p[0] for p in plan], [p[1] << (8 * p[5]) for p in plan],
                                      [p[2] for p in plan], [p[3] for p in plan], nslot=8 * nodes)
            rec["overlaps"], rec["feasible"] = ov, bool(ok)
        tab, optmap = R.table_from_tuples(tuples)
        bf = R.brute_force(tab, optmap, integer_starts=True, nodes=nodes)
        rec["bruteforce_int"] = {"makespan": bf[0], "opt": list(bf[1]), "prio": list(bf[2])}
        print(name, "status", rec["highs"].get("status"), "mk", rec.get("makespan"), "bf", bf[0],
              "overlaps", rec.get("overlaps"), "%.1fs" % rec["solver_wall_s"], flush=True)
        out["cases"].append(rec)
    dst = os.path.join(os.path.dirname(HERE), "tests", "golden", "milp_cases_n%d.json" % nodes)
    with open(dst, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", dst)


def main_forecast():
    """Fixtures for the interval loop: the reference's own forecast() (saturn/executor/executor.py:132-178)
    on duck-typed tasks; records its return values and the mutations it applies to the tasks."""
    milp, tight, Strategy, pulp = _load_reference()
    from saturn.executor import forecast           # the reference, unmodified (ray shim on sys.path)
    assert forecast.__code__.co_filename.startswith(REF)
    rnd = random.Random(5)
    out = {"generator": "oracle/gen_golden.py --forecast", "reference_commit": "b65e3d2", "cases": []}
    for case in range(6):
        J = rnd.randint(2, 7)
        interval = rnd.choice([100, 500, 1000])
        tasks, spec = [], []
        for t in range(J):
            base = rnd.uniform(50, 3000)
            opts = rnd.sample([1, 2, 4, 8], rnd.randint(1, 3))
            strategies = {g: Strategy("e", g, {}, base / g ** 0.8) for g in opts}
            task = DuckTask("t%d" % t, strategies)
            task.total_batches = rnd.randint(1, 400)
            task.select_strategy(strategies[rnd.choice(opts)])
            tasks.append(task)
            spec.append({"strategies": [[g, s.runtime] for g, s in strategies.items()],
                         "total_batches": task.total_batches,
                         "selected": task.selected_strategy.gpu_apportionment})
        starts = [float(rnd.choice([0, 0, rnd.randint(0, 2 * interval)])) for _ in range(J)]
        rel, btr, done = forecast(tasks, interval, starts)
        idx = {t: i for i, t in enumerate(tasks)}
        out["cases"].append({
            "interval": interval, "starts": starts, "tasks": spec,
            "relevant": [idx[t] for t in rel], "batches_to_run": [float(b) for b in btr],
            "completed": sorted(idx[t] for t in done),
            "after": [{"total_batches": t.total_batches,
                       "runtimes": [[g, s.runtime] for g, s in t.strategies.items()]} for t in tasks]})
    dst = os.path.join(os.path.dirname(HERE), "tests", "golden", "forecast_cases.json")
    with open(dst, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", dst, len(out["cases"]), "cases")


def _extra_worker(job):
    """One extra instance in its own process (HiGHS is single-threaded; the pool runs cases side by side)."""
    name, tuples, timeout = job
    milp, tight, Strategy, pulp = _load_reference()
    sys.path.insert(0, os.path.dirname(HERE))
    from oracle import ref_eval as R
    rec = run_case(tight, Strategy, pulp, name, tuples, timeout)
    rec["variant"] = "tight_m"
    if rec["incumbent"]:
        plan = R.plan_from_arrays(tuples, rec["sta"], rec["tga"], rec["bss"], rec["bna"])
        ok, ov, mk = R.check_plan([p[0] for p in plan], [p[1] for p in plan], [p[2] for p in plan],
                                  [p[3] for p in plan])
        rec["overlaps"], rec["feasible"] = ov, bool(ok)
    rec["proven_optimal"] = bool(rec["highs"].get("status") == 0)
    tab, optmap = R.table_from_tuples(tuples)
    bf = R.brute_force(tab, optmap, integer_starts=True)
    rec["bruteforce_int"] = {"makespan": bf[0], "opt": list(bf[1]), "prio": list(bf[2])}
    bf = R.brute_force(tab, optmap, integer_starts=False)
    rec["bruteforce_real"] = {"makespan": bf[0], "opt": list(bf[1]), "prio": list(bf[2])}
    print(name, "status", rec["highs"].get("status"), "mk", rec.get("makespan"), "bf",
          rec["bruteforce_int"]["makespan"], "overlaps", rec.get("overlaps"), "%.1fs" % rec["solver_wall_s"],
          flush=True)
    return rec


def main_extra():
    """Round 2: a thicker pin for SURVEY H6 (the list-schedule candidate space contains a MILP optimum):
    heterogeneous J = 4..5 instances and J = 6 instances, tight-M reference MILP with long HiGHS limits
    (run offline, several instances side by side) -> tests/golden/milp_cases_extra.json."""
    import multiprocessing as mp
    jobs = []
    if "--part3" in sys.argv:
        # more J = 6 (and a few J = 5) instances of the shapes HiGHS closes: H6 at the largest size it can prove
        for i, opts in enumerate(([8], [8], [8], [4, 8], [4, 8], [4, 8], [2, 8], [2, 8], [1, 8], [1, 8], [2, 4])):
            jobs.append(("J6_g%s_seed%d" % ("".join(map(str, opts)), 100 + i), probe_tuples(6, opts, 100 + i), 1200))
        for seed in range(110, 114):
            jobs.append(("H5_hetero_seed%d" % seed, hetero_tuples(5, seed), 1200))
        return _run_extra(jobs, "milp_cases_extra3.json", "--extra --part3")
    if "--part2" in sys.argv:
        # instances of the sizes HiGHS closes to a zero gap within minutes: more proven optima for H6
        for seed in range(50, 62):
            jobs.append(("H4_hetero_seed%d" % seed, hetero_tuples(4, seed), 420))
        for i, opts in enumerate(([1, 2], [2, 4], [4, 8], [2, 8], [1, 8], [1, 4])):
            jobs.append(("J4_g%s_seed%d" % ("".join(map(str, opts)), 70 + i), probe_tuples(4, opts, 70 + i), 420))
        for i, opts in enumerate(([8], [4, 8], [2, 8])):
            jobs.append(("J5_g%s_seed%d" % ("".join(map(str, opts)), 80 + i), probe_tuples(5, opts, 80 + i), 420))
        return _run_extra(jobs, "milp_cases_extra2.json", "--extra --part2")
    for seed in range(21, 29):
        jobs.append(("H4_hetero_seed%d" % seed, hetero_tuples(4, seed), 600))
    for seed in range(31, 39):
        jobs.append(("H5_hetero_seed%d" % seed, hetero_tuples(5, seed), 900))
    jobs += [
        ("J6_g8_seed6", probe_tuples(6, [8], 6), 600),
        ("J6_g48_seed7", probe_tuples(6, [4, 8], 7), 900),
        ("J6_g28_seed8", probe_tuples(6, [2, 8], 8), 900),
        ("H6_hetero_seed41", hetero_tuples(6, 41), 900),
        ("H6_hetero_seed42", hetero_tuples(6, 42), 900),
        ("H6_hetero_seed43", hetero_tuples(6, 43), 900),
        ("J5_g1248_seed9", probe_tuples(5, [1, 2, 4, 8], 9), 900),
        ("J5_g124_seed10", probe_tuples(5, [1, 2, 4], 10), 900),
    ]
    return _run_extra(jobs, "milp_cases_extra.json", "--extra")


def _run_extra(jobs, fname, how):
    import multiprocessing as mp
    workers = int(os.environ.get("GEN_GOLDEN_WORKERS", "6"))
    with mp.get_context("spawn").Pool(workers) as pool:
        recs = pool.map(_extra_worker, jobs, chunksize=1)
    out = {"generator": "ORACLE_MIP_REL_GAP=0 oracle/gen_golden.py " + how, "reference_commit": "b65e3d2",
           "scipy": __import__("scipy").__version__, "cases": recs}
    dst = os.path.join(os.path.dirname(HERE), "tests", "golden", fname)
    with open(dst, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", dst, "proven optimal:", sum(r["proven_optimal"] for r in recs), "of", len(recs))


def main_rerun(fname, name):
    """Re-run ONE recorded instance (its own gpu_time_tuples) under the current environment and replace the
    record.  Used with ORACLE_BIG_M_FACTOR=8 for instances where M = H + 1 over-tightens constraint family (iii)
    (milp.py:233-256: the rows of a NON-selected option with fewer GPUs need (k_sel / k' - 1) * start of slack,
    up to 7 H): there the tight-M MILP's "optimum" is worse than the true one; 8 (H + 1) is sound for all four
    families and still small enough for HiGHS' integrality tolerance (the overlap checker confirms)."""
    dst = os.path.join(os.path.dirname(HERE), "tests", "golden", fname)
    with open(dst) as f:
        d = json.load(f)
    for i, rec in enumerate(d["cases"]):
        if rec["name"] == name and rec["variant"] == "tight_m":
            tuples = [[tuple(x) for x in t] for t in rec["gpu_time_tuples"]]
            new = _extra_worker((name, tuples, 900))
            new["big_m_factor"] = float(os.environ.get("ORACLE_BIG_M_FACTOR", "1"))
            new["superseded"] = {"big_m_factor": 1.0, "makespan": rec.get("makespan"),
                                 "proven_optimal": rec.get("proven_optimal"),
                                 "why": "M = H + 1 cut off the optimum through constraint family (iii)"}
            d["cases"][i] = new
            with open(dst, "w") as f:
                json.dump(d, f, indent=1)
            print("replaced", name, "in", dst)
            return
    raise SystemExit("no such case")


def main_layout():
    """The reference's `saturn` package as data: every module file and the top-level functions it defines.
    tests/test_host_logic.py rebuilds an empty-bodied stand-in distribution from it to check the alias
    package's fall-through without the reference installed."""
    import ast
    modules, functions = [], {}
    for dirpath, dirnames, files in os.walk(os.path.join(REF, "saturn")):
        dirnames.sort()
        for f in sorted(files):
            if f.endswith(".py"):
                path = os.path.join(dirpath, f)
                rel = os.path.relpath(path, REF)
                modules.append(rel)
                with open(path) as fh:
                    names = [n.name for n in ast.parse(fh.read()).body if isinstance(n, ast.FunctionDef)]
                if names:
                    functions[rel] = names
    out = {"generator": "oracle/gen_golden.py --layout", "reference_commit": "b65e3d2", "modules": modules,
           "functions": functions}
    dst = os.path.join(os.path.dirname(HERE), "tests", "golden", "reference_layout.json")
    with open(dst, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", dst, len(modules), "modules")


def main():
    if "--layout" in sys.argv:
        return main_layout()
    if "--rerun" in sys.argv:
        i = sys.argv.index("--rerun")
        return main_rerun(sys.argv[i + 1], sys.argv[i + 2])
    if "--extra" in sys.argv:
        return main_extra()
    if "--forecast" in sys.argv:
        return main_forecast()
    if "--nodes" in sys.argv:
        return main_nodes(int(sys.argv[sys.argv.index("--nodes") + 1]))
    milp, tight, Strategy, pulp = _load_reference()
    sys.path.insert(0, os.path.dirname(HERE))
    from oracle import ref_eval as R

    cases = [
        ("K1_J3_g8_seed1", probe_tuples(3, [8], 1), 60),
        ("C1_J4_g12_seed0", probe_tuples(4, [1, 2], 0), 60),
        ("J3_g1248_seed0", probe_tuples(3, [1, 2, 4, 8], 0), 120),
        ("J4_g1248_seed3", probe_tuples(4, [1, 2, 4, 8], 3), 240),
        ("J4_g48_seed5", probe_tuples(4, [4, 8], 5), 120),
        ("J5_g248_seed2", probe_tuples(5, [2, 4, 8], 2), 240),
        ("H4_hetero_seed7", hetero_tuples(4, 7), 120),
        ("H5_hetero_seed11", hetero_tuples(5, 11), 240),
        ("K2_J5_g1248_seed0", probe_tuples(5, [1, 2, 4, 8], 0), 60),
    ]
    out = {"generator": "oracle/gen_golden.py", "reference_commit": "b65e3d2",
           "scipy": __import__("scipy").__version__, "cases": []}
    for name, tuples, timeout in cases:
        for variant, mod in (("tight_m", tight), ("as_shipped", milp)):
            rec = run_case(mod, Strategy, pulp, name, tuples, timeout if variant == "tight_m" else min(timeout, 60))
            rec["variant"] = variant
            if rec["incumbent"]:
                plan = R.plan_from_arrays(tuples, rec["sta"], rec["tga"], rec["bss"], rec["bna"])
                ok, ov, mk = R.check_plan([p[0] for p in plan], [p[1] for p in plan],
                                          [p[2] for p in plan], [p[3] for p in plan])
                rec["overlaps"] = ov
                rec["feasible"] = bool(ok)
            rec["proven_optimal"] = bool(rec["highs"].get("status") == 0)
            # exhaustive list-scheduling optimum for the same instance (oracle side)
            tab, optmap = R.table_from_tuples(tuples)
            bf = R.brute_force(tab, optmap, integer_starts=True)
            rec["bruteforce_int"] = {"makespan": bf[0], "opt": list(bf[1]), "prio": list(bf[2])}
            bf = R.brute_force(tab, optmap, integer_starts=False)
            rec["bruteforce_real"] = {"makespan": bf[0], "opt": list(bf[1]), "prio": list(bf[2])}
            print(name, variant, "status", rec["highs"].get("status"), "mk", rec.get("makespan"),
                  "bf", rec["bruteforce_int"]["makespan"], "overlaps", rec.get("overlaps"),
                  "%.1fs" % rec["solver_wall_s"], flush=True)
            out["cases"].append(rec)
    dst = os.path.join(os.path.dirname(HERE), "tests", "golden", "milp_cases.json")
    with open(dst, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", dst)


if __name__ == "__main__":
    main()
