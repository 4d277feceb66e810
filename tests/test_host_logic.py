"""CPU: host-side mirror of the reference interface (no GPU, no compute calls into the library)."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import DuckTask, build_c_host, tasks_from_tuples
from oracle import ref_eval as R
from saturn_b200 import HParams, Strategy, Task, Techniques, _lib
from saturn_b200.orchestrator import forecast
from saturn_b200.solver import (build_table, candidate_from_arrays, convert_into_comprehensible, gpu_time_tuples_of,
                                plan_to_arrays)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "saturn_b200.h")).read()
    declared = set(re.findall(r"^(?:int|const char\*)\s+(sb_[a-z0-9_]+)\s*\(", hdr, flags=re.M))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    lib = ctypes.CDLL(_lib.SO_PATH)
    for s in declared:
        assert hasattr(lib, s), s
    assert _lib.load().sb_abi_version() == 1


def test_header_is_plain_c_and_a_c_host_links(tmp_path):
    """include/saturn_b200.h compiles as C99 and a C host using only that header links against the library;
    without a GPU the host fails loudly at sb_create (no CPU path)."""
    import subprocess
    import torch
    exe = build_c_host(tmp_path)
    if not torch.cuda.is_available():
        r = subprocess.run([exe, "4"], capture_output=True, text=True)
        assert r.returncode == 1 and "no CPU path" in r.stderr


def test_ctypes_structs_match_the_header_layout(tmp_path):
    """The ctypes mirrors of the ABI's structs have the field offsets and sizes the C compiler gives them."""
    import subprocess
    structs = {"sb_search_params": _lib.SearchParams, "sb_search_control": _lib.SearchControl,
               "sb_search_result": _lib.SearchResultC}
    lines = []
    for cname, cls in structs.items():
        lines.append('printf("%s %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in cls._fields_:
            lines.append('printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "saturn_b200.h"\nint main(void) {\n%s\nreturn 0; }\n'
                   % "\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for cname, cls in structs.items():
        assert int(got[cname]) == ctypes.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got["%s.%s" % (cname, fname)]) == getattr(cls, fname).offset, (cname, fname)


def test_no_cpu_fallback_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = _lib.load()
    h = ctypes.c_void_p()
    rc = lib.sb_create(0, None, ctypes.byref(h))
    assert rc == -2 and not h.value                     # SB_ERR_CUDA
    assert b"no CPU path" in lib.sb_last_error()
    from saturn_b200.engine import Engine
    with pytest.raises(_lib.SaturnB200Error):
        Engine(0)
    from saturn_b200 import solve
    with pytest.raises(_lib.SaturnB200Error):
        solve(tasks_from_tuples([[(1, 10.0)], [(2, 5.0)]]))


def test_product_never_imports_oracle():
    """The product path may not import, link or execute anything under oracle/."""
    pat = re.compile(r"^\s*(from|import)\s+oracle\b|libref_eval|c_oracle|ref_eval\s*\(|ref_eval\.", re.M)
    for top in ("saturn_b200", "saturn"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h")):
                    src = open(os.path.join(dirpath, f)).read()
                    assert not pat.search(src), os.path.join(dirpath, f)


def test_representations_behave_like_reference():
    with pytest.raises(ValueError):
        Strategy(None, 0)
    with pytest.raises(ValueError):
        Strategy(None, 2.0)
    s = Strategy("ex", 4, {"a": 1}, 12.5)
    assert (s.executor, s.gpu_apportionment, s.parameters, s.runtime) == ("ex", 4, {"a": 1}, 12.5)
    assert str(s) == "Strategy(ex ({'a': 1}), 4G, 12.5s)"
    with pytest.raises(ValueError):
        HParams(0.1)
    with pytest.raises(ValueError):
        HParams(0.1, epochs=1, batch_count=3)
    assert HParams(0.1, epochs=2).as_dict() == {"lr": 0.1, "epochs": 2, "batch_count": None}
    assert [t.name for t in Techniques] == ["SPILLED", "PIPELINE", "FSDP", "MEGATRON"]


def test_task_object(tmp_path):
    t = Task(lambda: "model", lambda: list(range(10)), lambda a, b: 0.0, HParams(1e-3, epochs=3),
             save_dir=str(tmp_path / "ckpt"))
    assert t.epoch_length == 10 and t.total_batches == 30 and t.strategies == {} and t.selected_strategy is None
    assert len(t.name) == 16 and os.path.isdir(t.save_dir)
    t.reconfigure(13)
    assert t.current_batch == 3 and next(t.get_iterator()) == 3 and next(t.get_fresh_iterator()) == 0
    assert not t.has_ckpt() and t.get_model() == "model"
    t2 = Task(lambda kw: kw, lambda: [0], None, HParams(1e-3, batch_count=7, width=5), save_dir=str(tmp_path))
    assert t2.total_batches == 7 and t2.get_model() == {"width": 5}
    with pytest.raises(ValueError):
        Task(None, lambda: [0], None, HParams(1, epochs=1), hints={"is_transformer": True}, save_dir=str(tmp_path))
    s = Strategy("e", 2, None, 5.0)
    t.select_strategy(s)
    assert t.selected_strategy is s
    d = {t: 1}            # tasks are dict keys in the decoder's outputs (identity hash)
    assert d[t] == 1


def test_build_table_follows_dict_order_and_rounds_up():
    tasks = tasks_from_tuples([[(2, 10.1), (1, 30.0)], [(8, 7.0)], [(4, 1.0000001), (16, 0.5)]])
    assert gpu_time_tuples_of(tasks)[0] == [(2, 10.1), (1, 30.0)]
    T, usable, optindex = build_table(tasks)
    assert T.shape == (3, 1, 8) and T.dtype == np.float32
    assert optindex[0, 1] == 0 and optindex[0, 0] == 1 and optindex[1, 7] == 0
    assert optindex[2, 3] == 0 and (optindex[2] >= 0).sum() == 1           # 16 GPUs cannot fit a node
    assert float(T[0, 0, 1]) >= 10.1 and float(T[2, 0, 3]) >= 1.0000001    # fp32 rounded UP
    assert np.isinf(T[1, 0, 0])
    tasks[0].strategies[1].executor = None
    _, usable, _ = build_table(tasks)
    assert not usable[0, 0] and usable[0, 1]


def test_plan_arrays_satisfy_reference_constraints_and_decode():
    tuples = [[(1, 100.5), (2, 60.2)], [(2, 50.0)], [(8, 10.0), (4, 18.0)]]
    tasks = tasks_from_tuples(tuples)
    # plan: t0 on 2 GPUs {0,1} at 0; t1 on {2,3} at 0; t2 on all 8 at 61
    sta, tga, bss, bna, boa = plan_to_arrays([2, 1, 2], [1, 0, 0], [0.0, 0.0, 61.0], [0b11, 0b1100, 0xff], [0, 1, 2])
    assert R.milp_constraints_hold(tuples, sta, tga, bss, bna, boa, 71.0) == []
    assert R.milp_constraints_hold(tuples, sta, tga, bss, bna, boa, 70.0) != []      # makespan too small
    assert all(isinstance(v, float) for n in sta for g in n for v in g)
    assert boa[0][0] is None and boa[0][2] == 1.0 and boa[2][0] == 0.0
    npt, tdd, st = convert_into_comprehensible(tasks, bss, boa, tga, bna, sta)
    assert [npt[t] for t in tasks] == [0, 0, 0] and st == [0.0, 0.0, 61.0]
    assert tdd[tasks[2]] == [tasks[0], tasks[1]] and tasks[0] not in tdd and tasks[1] not in tdd
    assert tasks[0].selected_strategy.gpu_apportionment == 2 and tasks[2].selected_strategy.gpu_apportionment == 8
    # an overlapping plan is rejected by the restated constraints
    sta2, tga2, bss2, bna2, boa2 = plan_to_arrays([2, 1, 2], [1, 0, 0], [0.0, 0.0, 30.0], [0b11, 0b1100, 0xff],
                                                  [0, 1, 2])
    assert R.milp_constraints_hold(tuples, sta2, tga2, bss2, bna2, boa2, 100.0) != []
    warm = candidate_from_arrays(tasks, (sta, tga, bss, bna, boa, 71.0))
    assert list(warm[0]) == [1, 1, 7] and list(warm[1]) == [0, 1, 2]
    assert candidate_from_arrays(tasks[:2], (sta, tga, bss, bna, boa, 71.0)) is None


def test_decoder_matches_reference_decoder_on_reference_arrays(golden):
    """convert_into_comprehensible on the arrays the reference MILP returned must reproduce what the
    reference's own decoder (milp.py:448-513, run unmodified when the fixtures were generated) produced."""
    n = 0
    for rec in golden["cases"]:
        if not rec["incumbent"]:
            continue
        tasks = tasks_from_tuples(rec["gpu_time_tuples"])
        npt, tdd, st = convert_into_comprehensible(tasks, rec["bss"], rec["boa"], rec["tga"], rec["bna"], rec["sta"])
        d = rec["decoded"]
        assert [int(npt[t]) for t in tasks] == d["node_per_task"]
        assert [float(s) for s in st] == d["start"]
        idx = {t: i for i, t in enumerate(tasks)}
        assert [sorted(idx[x] for x in tdd[t]) for t in tasks] == d["deps"]
        assert [t.selected_strategy.gpu_apportionment for t in tasks] == d["selected_gpus"]
        n += 1
    assert n >= 10


def test_forecast_restates_executor_semantics():
    tasks = tasks_from_tuples([[(1, 1000.0), (2, 600.0)], [(2, 3000.0)], [(1, 100.0)]])
    for t in tasks:
        t.total_batches = 100
        t.select_strategy(list(t.strategies.values())[0])
    rel, btr, done = forecast(tasks, 500, [0.0, 100.0, 700.0])
    assert rel == tasks[:2]
    assert btr == [50.0, 13.0]            # 500 // 10 ; 400 // 30
    assert done == set()
    assert tasks[0].strategies[1].runtime == pytest.approx(500.0) and tasks[0].strategies[2].runtime == pytest.approx(300.0)
    assert tasks[0].total_batches == 50 and tasks[1].total_batches == 87
    assert tasks[2].total_batches == 100 and tasks[2].strategies[1].runtime == 100.0
    rel, btr, done = forecast(tasks, 1000, [0.0, 0.0, 0.0])
    assert tasks[0] in done and tasks[2] in done and tasks[1] not in done


def test_alias_package_paths():
    import saturn
    import saturn.solver
    import saturn.core.representations as rep
    import saturn.executor
    from saturn_b200 import solver
    assert saturn.solver.solve is solver.solve and saturn.solver.convert_into_comprehensible is solver.convert_into_comprehensible
    assert rep.Task is Task and rep.Strategy is Strategy and callable(saturn.orchestrate)


def test_product_and_oracle_generate_the_same_workload():
    from saturn_b200.synth import synth_table
    for (J, S, G, seed) in [(4, 2, 2, 0), (64, 6, 8, 0), (256, 8, 8, 0)]:
        a, va = synth_table(J, S, G, seed)
        b, vb = R.synth_table(J, S, G, seed)
        assert np.array_equal(a, b) and np.array_equal(va, vb)


def test_multi_node_plan_arrays_and_decoder(golden_n2):
    # emission: two nodes, tasks 0,1 on node 0 and task 2 on node 1
    tuples = [[(8, 100.0)], [(4, 30.5), (8, 20.0)], [(8, 70.0)]]
    tasks = tasks_from_tuples(tuples)
    sta, tga, bss, bna, boa = plan_to_arrays([1, 2, 1], [0, 0, 0], [0.0, 100.0, 0.0], [0xff, 0x0f, 0xff], [0, 2, 1],
                                             nodes=2, node_of=[0, 0, 1])
    assert len(sta) == 2 and bna == [[1.0, 0.0], [1.0, 0.0], [0.0, 1.0]]
    assert R.milp_constraints_hold(tuples, sta, tga, bss, bna, boa, 130.5) == []
    npt, tdd, st = convert_into_comprehensible(tasks, bss, boa, tga, bna, sta)
    assert [int(npt[t]) for t in tasks] == [0, 0, 1] and st == [0.0, 100.0, 0.0]
    assert tdd[tasks[1]] == [tasks[0]] and tasks[2] not in tdd
    warm = candidate_from_arrays(tasks, (sta, tga, bss, bna, boa, 130.5), nodes=2)
    assert list(warm[0]) == [7, 3, 7 | 8]
    # decoder parity on the arrays the reference MILP returned with 2 nodes
    for rec in golden_n2["cases"]:
        tasks = tasks_from_tuples(rec["gpu_time_tuples"])
        npt, tdd, st = convert_into_comprehensible(tasks, rec["bss"], rec["boa"], rec["tga"], rec["bna"], rec["sta"])
        d = rec["decoded"]
        idx = {t: i for i, t in enumerate(tasks)}
        assert [int(npt[t]) for t in tasks] == d["node_per_task"] and [float(x) for x in st] == d["start"]
        assert [sorted(idx[x] for x in tdd[t]) for t in tasks] == d["deps"]


def test_forecast_matches_reference_forecast():
    """forecast() against the reference's own forecast (executor.py:132-178) run unmodified when the
    fixtures were generated: same tasks launched, same batch counts, same completed set, and the same
    in-place mutations of every strategy runtime and of total_batches."""
    import json
    d = json.load(open(os.path.join(ROOT, "tests", "golden", "forecast_cases.json")))
    assert len(d["cases"]) >= 5
    for case in d["cases"]:
        tasks = []
        for t, spec in enumerate(case["tasks"]):
            task = DuckTask("t%d" % t, {int(g): Strategy("e", int(g), {}, float(rt)) for g, rt in spec["strategies"]},
                            total_batches=spec["total_batches"])
            task.select_strategy(task.strategies[spec["selected"]])
            tasks.append(task)
        rel, btr, done = forecast(tasks, case["interval"], case["starts"])
        idx = {t: i for i, t in enumerate(tasks)}
        assert [idx[t] for t in rel] == case["relevant"]
        assert [float(b) for b in btr] == case["batches_to_run"]
        assert sorted(idx[t] for t in done) == case["completed"]
        for task, after in zip(tasks, case["after"]):
            assert task.total_batches == after["total_batches"]
            assert [[g, s.runtime] for g, s in task.strategies.items()] == after["runtimes"]


# ------------------------------------------------------------------------------------------ round 2
def test_alias_package_falls_through_to_an_installed_reference(tmp_path):
    """`import saturn` is this repository's alias; submodules it does not implement resolve in a reference
    distribution when one is on sys.path (saturn_b200/_alias.py) and raise a clear ImportError otherwise.
    The reference is a stand-in with the reference package's module layout (tests/golden/reference_layout.json):
    every module file exists and each top-level function returns the path of the file that defines it."""
    import json
    import subprocess
    import sys
    with open(os.path.join(ROOT, "tests", "golden", "reference_layout.json")) as f:
        layout = json.load(f)
    ref = tmp_path / "reference"
    for rel in layout["modules"]:
        path = ref / rel
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_text("".join("def %s(*args, **kwargs):\n    return %r\n" % (name, rel)
                                for name in layout["functions"].get(rel, [])))
    code = r'''
import sys
sys.path.insert(0, %r)
import saturn, saturn.solver, saturn.core.representations as Rp, saturn.executor as E
assert saturn.solver.solve.__module__ == "saturn_b200.solver"
assert Rp.Task.__module__ == "saturn_b200.representations"
try:
    import saturn.library
    raise SystemExit("saturn.library must not resolve without a reference distribution")
except ImportError:
    pass
try:
    E.execute
    raise SystemExit("saturn.executor.execute must not resolve without a reference distribution")
except ImportError as e:
    assert "not part of the B200 solver drop-in" in str(e)
ref = %r
sys.path.append(ref)
for m in [m for m in sys.modules if m == "saturn" or m.startswith("saturn.")]:
    del sys.modules[m]
import saturn, saturn.solver, saturn.library, saturn.core.representations as Rp, saturn.executor as E
assert saturn.library.__file__.startswith(ref)                      # fell through
assert saturn.solver.solve.__module__ == "saturn_b200.solver"       # the drop-in still wins
assert saturn.orchestrate.__module__ == "saturn_b200.orchestrator"
assert E.execute() == "saturn/executor/executor.py"                 # names the drop-in lacks come from the reference
assert Rp.search() == "saturn/core/representations/Strategy.py"
print("ok")
''' % (ROOT, str(ref))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr


def _profiler_reduction(n_tasks, executors, gpu_ranges, flat, max_gpus):
    """PerformanceEvaluator.py:96-115 restated literally on (executor name, params, runtime) tuples."""
    out = []
    idx = 0
    for t in range(n_tasks):
        d = {g: (None, None, 1000000) for g in range(1, max_gpus + 1)}               # :96-99
        rng_t = gpu_ranges[t] if gpu_ranges[t] is not None else list(range(1, max_gpus + 1))
        for g in rng_t:
            chosen = (None, None, 1e8)                                                   # :106
            for e in executors:
                params, runtime = flat[idx]
                idx += 1
                if params is not None and runtime < chosen[2]:                            # :109-110
                    chosen = (e, params, runtime)
            d[g] = chosen
        out.append(d)
    return out


def test_dense_table_from_trials_matches_the_profiler_reduction():
    """table_from_trials + strategies_from_table == the dict the trial runner attaches to every task
    (PerformanceEvaluator.py:96-115): fastest executor per GPU count, first minimum on ties, 1e6 where the
    count is outside the task's gpu_range, 1e8 / executor None where every executor failed."""
    from saturn_b200.solver import FAILED, NOT_PROFILED, strategies_from_table, table_from_trials
    rng = np.random.default_rng(4)
    executors = ["spill", "ddp", "fsdp"]
    n_tasks, G = 7, 8
    gpu_ranges = [None, [1, 2, 4], [2, 4, 8], None, [8], [1], [3, 5, 6]]
    flat = []
    for t in range(n_tasks):
        for g in (gpu_ranges[t] or range(1, G + 1)):
            for e in range(len(executors)):
                if rng.uniform() < 0.3:
                    flat.append((None, None))
                else:
                    flat.append(({"bs": int(rng.integers(1, 9))}, float(np.float32(rng.uniform(100, 5000)))))
    flat[0] = ({"bs": 1}, 777.0)
    flat[1] = ({"bs": 2}, 777.0)                  # a tie: the first executor must win
    flat[2] = (None, None)
    T, mask, params = table_from_trials(n_tasks, len(executors), gpu_ranges, flat, max_gpus=G)
    assert T.shape == mask.shape == (n_tasks, len(executors), G) and T.dtype == np.float32
    got = strategies_from_table(T, mask, executors, params)
    want = _profiler_reduction(n_tasks, executors, gpu_ranges, flat, G)
    for t in range(n_tasks):
        assert list(got[t].keys()) == list(range(1, G + 1))
        for g in range(1, G + 1):
            e, prm, rt = want[t][g]
            s = got[t][g]
            assert s.executor == e and s.gpu_apportionment == g
            assert s.runtime == pytest.approx(rt, rel=1e-6) and (s.parameters == prm)
    assert got[0][1].executor == "spill" and got[0][1].runtime == 777.0
    assert (T[~mask] >= NOT_PROFILED).all() and set(np.unique(T[~mask])) <= {np.float32(NOT_PROFILED), np.float32(FAILED)}
    # the oracle's device-side statement of the same reduction (first minimum over strategies)
    tab = R.canon_table(np.where(mask, T, np.inf), range(1, G + 1))
    tmin, args = R.reduce_table(tab)
    for t in range(n_tasks):
        for g in range(1, G + 1):
            if mask[t, :, g - 1].any():
                assert tmin[t, g - 1] == np.float32(got[t][g].runtime)
                assert executors[int(args[t, g - 1])] == got[t][g].executor


def test_fp32_horizon_guard():
    """Schedule times are exact integers in fp32 only below 2^24 s: a table that can cross it is refused."""
    from saturn_b200.solver import SolverError, _check_horizon
    T = np.full((200, 1, 8), np.inf, dtype=np.float32)
    T[:, 0, 0] = 1.0e6                     # 200 jobs of 1e6 s on one GPU each: area bound 2.5e7 s > 2^24
    with pytest.raises(SolverError):
        _check_horizon(T)
    T[:, 0, 0] = 36000.0
    _check_horizon(T)
    _check_horizon(T, found_makespan=1.5e7)
    with pytest.raises(SolverError):
        _check_horizon(T, found_makespan=float(1 << 24))
