#!/usr/bin/env python
"""bench.py — candidate schedules evaluated / second on the SPASE hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic candidates per GPU:
  sb_eval (k_eval_tiles) over B candidates of the BASELINE C4 workload (J=256 jobs, S=8
  strategies, G=1..8 GPUs; configs[3] of BASELINE.json, which fits one GPU), folding the 64-bit
  arg-min key, and — for N > 1 — the one exchange the path has: a MIN of that key over all ranks.
  Default: NVLink peer memory, fused into the evaluation kernel (publish in its tail, fold of the previous
  step's keys between its tiles, last step folded by a one-warp kernel inside the timed region);
  SATURN_B200_EXCHANGE=nccl (or peers that cannot be mapped) falls back to one NCCL all_reduce(MIN) per
  step.  Candidates shard by id, no data-path collective.  Weak scaling: B per GPU is fixed.

`value`  = candidates scored by all ranks / device time of the K steps (inputs resident in HBM).
`e2e`    = same metric, same batch, through the public host-buffer call (Engine.eval_host -> sb_eval_host):
           candidate encodings start in pinned HOST memory, H2D + kernel + D2H of the makespans
           inside the timed region.
`roofline` = algorithmic bytes (J*(1+w)+4 per candidate, SURVEY §8d) of one k_eval_tiles launch /
           its CUDA-event duration, against the measured HBM copy bandwidth.
`cpu_baseline` / `--impl reference` = oracle/cpu_arm.py: the oracle's C restatement (oracle/ref_eval.c,
           kind "port") on the physical host cores, run in its own process; both legs are the same function.
`milp`   = the reference's CPU MILP (oracle/ref_milp.py, HiGHS, time-limited) on J = 8 and 16 next to
           saturn.solver.solve() on the same T: time for the GPU search to match the MILP's makespan; for
           C4 the MILP cannot be built (row count reported) and the GPU plan is held to the area lower bound.
`configs` = the other BASELINE shapes (C3, C5) as short diagnostic runs; `exchange_check` (N > 1) = the
           peer-memory MIN re-derived with an NCCL all_reduce(MIN) outside the timed region.

--dump-outputs DIR writes what the last timed step returned to its caller (rank 0): DIR/makespan.npy (fp32, one
per candidate), DIR/candidate_id.npy (fp64, the global id of each of those candidates) and the folded arg-min key
as DIR/best_makespan.npy (fp32) + DIR/best_candidate_id.npy (fp64).  Inputs are seeded, so two builds run with the
same arguments can be compared output for output.  Batches above DUMP_CANDIDATES are sampled (fixed seed).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "candidate schedules/sec"
UNIT = "candidates/s"
J, S, G = 256, 8, 8
WORKLOAD = "C4: J=256 jobs x S=8 strategies x G=1..8 GPUs, synthetic T (seed 0), integer starts"
WAVE = 148 * 8 * 32           # candidates in one half wave of 32-candidate tiles (148 SMs x 16 resident warps / 2)
B_PER_GPU = WAVE * 28         # 1,060,864 candidates = 14 whole tiles for every resident warp of the persistent
                              # grid (no idle warps in a last partial wave) = 543 MB of encodings per step (> 126 MB L2)
FALLBACK_HBM_GBS = 6650.0
DUMP_CANDIDATES = 1 << 22     # at most 48 MB of dumped makespans + ids


def bytes_per_candidate(j):
    w = 1 if j <= 256 else 2
    return j * (1 + w) + 4


class ClockSampler:
    """nvidia-smi sampler running during the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """dram bytes per k_eval_tiles launch from the committed ncu --set full capture, if any."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(p) as f:
            d = json.load(f)
        return d.get("dram_bytes_per_launch"), d.get("candidates_per_launch")
    except Exception:
        return None, None


def static_config(ints=True, config="C4"):
    """The `config` object both arms print (identical for the same run shape, so the driver's same_config holds)."""
    return {"workload": WORKLOAD, "integer_starts": bool(ints),
            "l2": "no flush needed: every step streams its whole input once — GPU arm %.0f MB of candidate encodings "
                  "per GPU per step (> 126 MB L2); CPU arm >= 2 M candidate evaluations per step" % (
                      B_PER_GPU * 2 * 256 / 1e6)}


def _clean_env():
    env = dict(os.environ)
    for k in ("OMP_NUM_THREADS", "OMP_PROC_BIND", "OMP_PLACES", "MKL_NUM_THREADS", "GOMP_CPU_AFFINITY", "KMP_AFFINITY"):
        env.pop(k, None)                  # torchrun pins OMP_NUM_THREADS=1; the CPU arm picks its own thread count
    return env


def cpu_arm(steps, warmup, config="C4", timeout=900, all_steps=False):
    """oracle/cpu_arm.py in its own process (before / without torch): the one CPU measurement both the
    `cpu_baseline` leg and `--impl reference` report.  all_steps: time every one of the `steps` steps (no
    time cap)."""
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "cpu_arm.py"), "--steps", str(steps), "--warmup", str(warmup),
           "--config", config] + (["--max-seconds", "inf"] if all_steps else [])
    out = subprocess.run(cmd, env=_clean_env(), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout)
    if out.returncode != 0:
        raise RuntimeError("oracle/cpu_arm.py failed: %s" % out.stderr[-2000:])
    return json.loads(out.stdout.strip().splitlines()[-1])


def run_reference(args):
    """--impl reference: the CPU restatement of the path (oracle port) on all physical host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_arm(args.steps, args.warmup, timeout=None, all_steps=True)
    val = r["value"]
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": r["steps_timed"], "warmup": args.warmup, "ms_per_step": r["ms_per_step_median"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": static_config(True),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"]},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "run": {"candidates_per_step": r["candidates_per_step"], "ms_per_step_min": r["ms_per_step_min"],
                    "ms_per_step_max": r["ms_per_step_max"], "build": r["build"], "cores_how": r["cores_how"]},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, out, key, id_base):
    """The last timed step's outputs as .npy files (see the module docstring)."""
    from saturn_b200.search import key_makespan
    mk = out.cpu().numpy()
    ids = np.arange(mk.shape[0])
    if mk.shape[0] > DUMP_CANDIDATES:
        ids = np.sort(np.random.default_rng(0).choice(mk.shape[0], DUMP_CANDIDATES, replace=False))
    k = int(key.item())
    arrays = {"makespan": mk[ids].astype(np.float32), "candidate_id": (ids + id_base).astype(np.float64),
              "best_makespan": np.array([key_makespan(k)], dtype=np.float32),
              "best_candidate_id": np.array([k & 0xffffffff], dtype=np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class _Task:
    def __init__(self, name, strategies):
        self.name, self.strategies, self.selected_strategy = name, strategies, None

    def select_strategy(self, st_):
        self.selected_strategy = st_


def milp_leg_finish(proc, eng, c4_tasks, c4_plan_makespan, c4_wall):
    """Join the MILP subprocess and time saturn.solver.solve() on the same instances."""
    import random
    from saturn_b200 import Strategy, solve
    from saturn_b200 import solver as sb_solver
    from saturn_b200.search import run_search
    try:
        out, err = proc.communicate(timeout=240)
        milp = json.loads(out.strip().splitlines()[-1])
    except Exception as e:                                            # the baseline leg must not sink the bench line
        try:
            proc.kill()
        except Exception:
            pass
        return {"error": "milp leg failed: %r" % (e,)}
    for rec in milp["instances"]:
        J = rec["J"]
        rnd = random.Random(rec["seed"])
        tuples = [[(g, b / g ** 0.8) for g in milp["options"]] for b in (rnd.uniform(500, 4000) for _ in range(J))]
        tasks = [_Task("t%d" % t, {g: Strategy("x", g, {}, rt) for g, rt in tup}) for t, tup in enumerate(tuples)]
        t0 = time.perf_counter()
        plan = solve(tasks, None, engine=eng, chains=1 << 16, rounds=200)
        rec["gpu_solve_s"] = time.perf_counter() - t0
        rec["gpu_makespan"] = plan[5]
        rec["gpu_candidates"] = sb_solver.last_stats["candidates"]
        if rec["makespan"] is not None:
            # time to match: table upload + search until the incumbent is <= the MILP's makespan
            T, usable, _oi = sb_solver.build_table(tasks)
            Td = np.where(usable[:, None, :], T, np.inf).astype(np.float32)
            t0 = time.perf_counter()
            eng.set_table(Td, list(range(1, 9)), sentinel=float("inf"))
            res = run_search(eng, chains=1 << 16, rounds=400, seed=0, reduced=True, time_budget_s=10.0,
                             target_makespan=float(np.float32(rec["makespan"] * (1 + 1e-6))), use_dist=False)
            dt = time.perf_counter() - t0
            rec["gpu_time_to_match_s"] = dt if res.makespan <= rec["makespan"] * (1 + 1e-5) else None
            rec["gpu_rounds_to_match"] = res.rounds
            rec["milp_over_gpu_makespan"] = rec["makespan"] / plan[5]
            rec["speedup_to_match"] = (rec["wall_s"] / dt) if rec["gpu_time_to_match_s"] else None
    # C4: the MILP cannot be built; the GPU plan is held to the area lower bound sum_j min_k(k * rt_jk) / 8
    lb = sum(min(g * st_.runtime for g, st_ in t.strategies.items()) for t in c4_tasks) / 8.0
    milp["c4"] = dict(milp.pop("c4_model"), gpu_makespan=c4_plan_makespan, gpu_solve_s=c4_wall,
                      area_lower_bound=lb, gap_to_lower_bound=c4_plan_makespan / lb - 1.0)
    return milp


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 200; 5 for --impl reference)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=B_PER_GPU, help="candidates per GPU per step")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline and milp legs")
    ap.add_argument("--no-e2e", action="store_true", help="skip the e2e / solve_api / search_round / configs legs")
    ap.add_argument("--no-milp", action="store_true")
    ap.add_argument("--real", action="store_true", help="real-valued starts instead of integer starts")
    ap.add_argument("--config", default="C4", choices=["C2", "C3", "C4", "C5"],
                    help="BASELINE config shape (C4 is the headline; the others are diagnostic runs)")
    ap.add_argument("--reduced", action="store_true", help="evaluate on the min-over-strategies table")
    ap.add_argument("--solve-devices", type=int, default=0,
                    help="N = 1 only, opt-in: also time saturn.solver.solve(..., devices=D) — ONE process driving D GPUs "
                         "(it touches GPUs beyond --gpus, so it is never run by default)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to --impl ours")
        if args.steps is None:
            args.steps = 5                                            # default K for the CPU arm: minutes, not hours
        return run_reference(args)
    if args.steps is None:
        args.steps = 200
    args.warmup = max(args.warmup, 3)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    headline = args.config == "C4" and not args.reduced
    # the MILP leg is CPU work on one core: start it now, it runs beside the GPU legs (rank 0, N = 1)
    milp_proc = None
    if rank == 0 and world == 1 and headline and not (args.no_cpu or args.no_milp or args.no_e2e):
        milp_proc = subprocess.Popen([sys.executable, os.path.join(ROOT, "oracle", "milp_leg.py"), "--sizes", "8,16",
                                      "--limit", "12"], env=_clean_env(), stdout=subprocess.PIPE,
                                     stderr=subprocess.PIPE, text=True)

    import torch
    import torch.distributed as dist
    from saturn_b200.synth import synth_table
    from saturn_b200.engine import Engine, opt_by_position, random_candidates

    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun (one process per GPU)" % args.gpus)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ints = not args.real

    eng = Engine(local)
    global J, S, G, WORKLOAD
    if args.config != "C4":
        from saturn_b200.synth import CONFIGS
        J, S, G, _seed = CONFIGS[args.config]
        WORKLOAD = "%s: J=%d jobs x S=%d strategies x G=1..%d GPUs, synthetic T (diagnostic, not the headline)" % (
            args.config, J, S, G)
        if args.batch == B_PER_GPU:
            args.batch = max(2 * WAVE, (B_PER_GPU * 256 // J) // (2 * WAVE) * (2 * WAVE))
    T, valid = synth_table(J, S, G, seed=0)
    if args.reduced:
        T = np.where(valid, T, np.inf).min(axis=1, keepdims=True).astype(np.float32)
        valid = np.isfinite(T)
        T = np.where(valid, T, 1e8).astype(np.float32)
    eng.set_table(T)
    B = args.batch
    opt, prio = random_candidates(eng, B, valid, seed=1 + rank)
    out = torch.empty(B, dtype=torch.float32, device=dev)
    KEY_MAX = 2 ** 63 - 1
    key = torch.full((1,), KEY_MAX, dtype=torch.int64, device=dev)
    id_base = (rank * B) & 0xffffffff

    # the per-step exchange: NVLink peer-memory MIN (post fused into the evaluation kernel's tail, fold of the
    # previous step between its tiles), falling back to one NCCL all-reduce of the key if the IPC mappings
    # cannot be opened — xchg_init decides collectively
    use_xchg = False
    if world > 1 and os.environ.get("SATURN_B200_EXCHANGE", "peer") == "peer":
        use_xchg = eng.xchg_init(dist)
    gmin = torch.zeros(1, dtype=torch.int64, device=dev)
    pipelined = use_xchg and os.environ.get("SATURN_B200_EXCHANGE_PIPELINE", "1") != "0"

    def exchange_after_eval():
        if use_xchg:
            if not pipelined:
                eng.xchg_reduce(gmin, fold=key)             # the running best becomes the global one
        else:
            dist.all_reduce(key, op=dist.ReduceOp.MIN)

    def step():
        # pipelined: ONE kernel per step evaluates the batch, folds the keys every rank published in the
        # previous step (NVLink loads between its tiles) and publishes this step's key (tail)
        eng.eval(opt, prio, integer_starts=ints, out=out, best_key=key, id_base=id_base,
                 post_key=use_xchg, fold_prev=pipelined)
        if world > 1:
            exchange_after_eval()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rendezvous():
        # Device-side rendezvous queued right in front of the timed region (after the host barrier): every
        # rank's stream passes it within an NVLink round trip of the others, so the K timed steps start
        # together on all GPUs instead of up to a host-wake-up apart — the per-step fold makes ranks wait for
        # the slowest one, and with K = 20 a start skew of a fraction of a millisecond is a visible share of
        # the 9 ms timed region (round-1 SCALE: 0.918 at N = 8 with 20 steps, 0.989 with 200).
        if world > 1:
            if use_xchg:
                eng.xchg_post(key)
                eng.xchg_reduce(gmin)
            else:
                dist.all_reduce(gmin, op=dist.ReduceOp.MIN)

    for _ in range(args.warmup):
        step()
    barrier()
    if headline:
        assert eng.last_eval_path() == 3, "bench must run the TMA + streaming tile kernel"
    kernel_path = eng.last_eval_path()

    # ---- timed region: K steps, device time, max over ranks
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    k_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    rendezvous()
    e0.record()
    for i in range(args.steps):
        k_ev[i][0].record()
        eng.eval(opt, prio, integer_starts=ints, out=out, best_key=key, id_base=id_base, post_key=use_xchg,
                 fold_prev=pipelined)
        k_ev[i][1].record()
        if world > 1:
            exchange_after_eval()
    if pipelined:
        eng.xchg_reduce(gmin, fold=key)                     # fold the last step's keys inside the timed region
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if use_xchg:
        eng.xchg_check()
    ms_total = e0.elapsed_time(e1)
    per_step = np.array([a.elapsed_time(b) for a, b in k_ev])
    kern_ms = float(per_step.mean())
    t = torch.tensor([ms_total, kern_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total_max, kern_ms_max = float(t[0]), float(t[1])
    value = world * B * args.steps / (ms_total_max * 1e-3)
    rank_stats = torch.tensor([ms_total, float(per_step.min()), float(np.median(per_step)), float(per_step.max()),
                               float(per_step[0])], dtype=torch.float64, device=dev)
    all_stats = [torch.empty_like(rank_stats) for _ in range(world)]
    if world > 1:
        dist.all_gather(all_stats, rank_stats)
    else:
        all_stats = [rank_stats]
    per_rank = [{"rank": r, "timed_ms": float(x[0]), "kernel_ms_min": float(x[1]), "kernel_ms_median": float(x[2]),
                 "kernel_ms_max": float(x[3]), "kernel_ms_first": float(x[4])} for r, x in enumerate(all_stats)]
    if args.dump_outputs and rank == 0:                       # before any later leg reuses `out`
        dump_outputs(args.dump_outputs, out, key, id_base)

    # ---- N > 1, outside the timed region: the fused peer-memory MIN against NCCL's
    exchange_check = None
    if world > 1:
        # (a) the running key after the timed steps must be the same on every rank
        kk = key.clone()
        lo, hi = kk.clone(), kk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        same_everywhere = bool(lo.item() == hi.item() == kk.item())
        # (b) three fresh steps through the exchange vs the per-rank LOCAL keys (same deterministic batch, no
        #     exchange flags) reduced with one NCCL all_reduce(MIN)
        local_key = torch.full((1,), KEY_MAX, dtype=torch.int64, device=dev)
        eng.eval(opt, prio, integer_starts=ints, out=out, best_key=local_key, id_base=id_base)
        nccl_key = local_key.clone()
        dist.all_reduce(nccl_key, op=dist.ReduceOp.MIN)
        key.fill_(KEY_MAX)
        barrier()
        for _ in range(3):
            step()
        if pipelined:
            eng.xchg_reduce(gmin, fold=key)
        torch.cuda.synchronize()
        if use_xchg:
            eng.xchg_check()
        agree = torch.tensor([1 if int(key.item()) == int(nccl_key.item()) else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(agree, op=dist.ReduceOp.MIN)
        exchange_check = bool(agree.item()) and same_everywhere
        owner = (int(nccl_key.item()) & 0xffffffff) // B
        exchange_detail = {"folded_key": int(key.item()), "nccl_min_of_local_keys": int(nccl_key.item()),
                           "owner_rank": int(owner), "timed_key_identical_on_all_ranks": same_everywhere,
                           "path": "peer-memory mailboxes" if use_xchg else "nccl all_reduce"}

    # ---- e2e: host buffers through the public call, same batch as `value`
    e2e = None
    if not args.no_e2e:
        from saturn_b200.engine import padded_rows
        od, pd_ = random_candidates(eng, B, valid, seed=100 + rank)     # generated on the device, parked in pinned host memory
        oh, ph = padded_rows(B, J, torch.uint8, "cpu", pinned=True), padded_rows(B, J, eng.prio_dtype, "cpu", pinned=True)
        oh.copy_(od)
        ph.copy_(pd_)
        del od, pd_
        outh = torch.empty(B, dtype=torch.float32, pin_memory=True)
        e2e_steps = min(args.steps, 20)
        for _ in range(2):
            eng.eval_host(oh, ph, integer_starts=ints, out=outh)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            eng.eval_host(oh, ph, integer_starts=ints, out=outh)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt[0])
        stride = oh.stride(0)
        e2e = {"value": world * B * e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(B * stride * (1 + (1 if J <= 256 else 2))), "d2h_bytes_per_step": int(B * 4),
               "candidates_per_gpu_per_step": B, "steps": e2e_steps,
               "api": "saturn_b200.engine.Engine.eval_host -> sb_eval_host",
               "bound": "PCIe: %d B of encodings per candidate host->device" % (stride * (1 + (1 if J <= 256 else 2)))}
        del oh, ph, outh

    # ---- the reference-facing call itself: saturn.solver.solve(task_list) on host Task objects
    solve_leg = None
    c4_tasks = None
    if not args.no_e2e and headline:
        from saturn_b200 import Strategy, solve
        from saturn_b200 import solver as sb_solver
        tmin_h = np.where(valid, T, np.inf).min(axis=1)
        c4_tasks = [_Task("t%d" % j, {g + 1: Strategy("x", g + 1, {}, float(tmin_h[j, g])) for g in range(G)
                                      if np.isfinite(tmin_h[j, g])}) for j in range(J)]
        solve(c4_tasks, None, engine=eng, rounds=8)                  # warm-up
        barrier()
        t0 = time.perf_counter()
        plan = solve(c4_tasks, None, engine=eng, rounds=200)
        dt = time.perf_counter() - t0
        stt = dict(sb_solver.last_stats)
        solve_leg = {"value": stt["candidates"] / dt, "unit": UNIT, "wall_s": dt, "candidates": stt["candidates"],
                     "makespan": plan[5], "h2d_bytes": int(J * 8 * 4), "d2h_bytes": int(J * (8 + 4 + 1 + 1 + 1)),
                     "api": "saturn.solver.solve(task_list) -> (sta, tga, bss, bna, boa, makespan); per rank"}
        # one process, every GPU of the node: saturn.solver.solve(..., devices=N) (sb_search_run_multi)
        ndev = min(args.solve_devices, torch.cuda.device_count())
        if world == 1 and ndev > 1:
            solve(c4_tasks, None, devices=ndev, rounds=8)
            t0 = time.perf_counter()
            plan_n = solve(c4_tasks, None, devices=ndev, rounds=200)
            dtn = time.perf_counter() - t0
            sn = dict(sb_solver.last_stats)
            solve_leg["devices_%d" % ndev] = {"value": sn["candidates"] / dtn, "wall_s": dtn, "candidates": sn["candidates"],
                                             "makespan": plan_n[5], "speedup_vs_1_device": (sn["candidates"] / dtn) /
                                             (stt["candidates"] / dt)}

    # ---- one fused search round at a large population (diagnostic: the kernel the solver actually runs)
    search_leg = None
    if not args.no_e2e and headline:
        eng.set_table(T)
        wave = eng.search_wave(reduced=True)
        chains = wave * max(1, round((1 << 20) / wave))      # ~1 M chains in whole waves of the round kernel
        i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        i0.record()
        eng.search_init(chains, seed=rank, chain_base=rank * chains, integer_starts=ints, reduced=True,
                        t_start=5e-4, t_end=1e-6, total_rounds=64)
        i1.record()
        eng.search_round(16)
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        eng.search_round(32)
        s1.record()
        torch.cuda.synchronize()
        ms = s0.elapsed_time(s1) / 32
        search_leg = {"candidates_per_s_per_gpu": chains / (ms * 1e-3), "ms_per_round": ms, "chains_per_gpu": chains,
                      "fused": eng.search_is_fused(), "rounds_per_launch": 16,
                      "init_ms": i0.elapsed_time(i1),
                      "what": "the round kernel solve() runs (min-over-strategies table): move + evaluate + Metropolis "
                              "accept of every chain, scored incrementally from the snapshot in front of the warp's move window, 16 rounds per "
                              "launch with the rows resident in shared memory; "
                              "init_ms = sb_search_init of that population (shuffle in shared memory + first scoring)"}

    # ---- the other BASELINE shapes, a fraction of a second each (diagnostic)
    configs = None
    if not args.no_e2e and headline and rank == 0:
        from saturn_b200.synth import CONFIGS
        peak_c, _src = measured_peak()
        configs = {}
        for name, by_pos, reduced_c in (("C3", False, False), ("C5", True, True), ("C5_full_table", False, False)):
            Jc, Sc, Gc, _sd = CONFIGS[name.split("_")[0]]
            Tc, vc = synth_table(Jc, Sc, Gc, seed=0)
            if reduced_c:                                    # J = 1024: the search's own view, 32 KB in shared memory
                vr = vc.any(axis=1, keepdims=True)
                eng.set_table(Tc)
                valid_c = vr
            else:
                eng.set_table(Tc)
                valid_c = vc
            Bc = max(2 * WAVE, (B_PER_GPU * 256 // Jc) // (2 * WAVE) * (2 * WAVE))      # whole waves of 16 warps per SM
            oc, pc = random_candidates(eng, Bc, valid_c, seed=11)
            if by_pos:
                oc = opt_by_position(oc, pc)
            outc = torch.empty(Bc, dtype=torch.float32, device=dev)
            for _ in range(2):
                eng.eval(oc, pc, integer_starts=ints, reduced=reduced_c, out=outc, by_position=by_pos)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            nrep = 8
            c0.record()
            for _ in range(nrep):
                eng.eval(oc, pc, integer_starts=ints, reduced=reduced_c, out=outc, by_position=by_pos)
            c1.record()
            torch.cuda.synchronize()
            msc = c0.elapsed_time(c1) / nrep
            gbs = Bc * bytes_per_candidate(Jc) / (msc * 1e-3) / 1e9
            configs[name] = {"J": Jc, "S": Sc, "candidates_per_launch": Bc, "ms_per_launch": msc,
                             "candidates_per_s": Bc / (msc * 1e-3), "achieved_GBps": gbs, "frac": gbs / peak_c,
                             "eval_path": eng.last_eval_path(),
                             "encoding": ("opt by schedule position, min-over-strategies table (the population "
                                          "encoding of the J > 512 search)" if by_pos else
                                          "job-indexed opt, full table" if name == "C3" else
                                          "job-indexed opt, all 8 strategies (256 KB of table): rows re-ordered on the "
                                          "device, position-major kernel reading the table through L1 (round 1: tile "
                                          "kernel path 4, 1.2e8)")}
            del oc, pc, outc
        # the kernel shape the north star sketches (slot times across lanes + warp shuffles), same C4 candidates
        eng.set_table(T)
        Ba = 4 * WAVE
        for _ in range(2):
            eng.eval(opt[:Ba], prio[:Ba], integer_starts=ints, out=out[:Ba], alt_shape=True)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(8):
            eng.eval(opt[:Ba], prio[:Ba], integer_starts=ints, out=out[:Ba], alt_shape=True)
        c1.record()
        torch.cuda.synchronize()
        msa = c0.elapsed_time(c1) / 8
        configs["C4_alt_shape"] = {"J": J, "S": S, "candidates_per_launch": Ba, "ms_per_launch": msa,
                                   "candidates_per_s": Ba / (msa * 1e-3), "eval_path": eng.last_eval_path(),
                                   "frac": Ba * bytes_per_candidate(J) / (msa * 1e-3) / 1e9 / peak_c,
                                   "encoding": "SB_FLAG_ALT_WARPSCAN: 8 lanes per candidate, 4 candidates per warp, the "
                                               "sorted slot times shifted with shuffles — measured for comparison with "
                                               "the shipped lane-per-candidate kernel (`value`), not used"}
        eng.set_table(T)

    if rank == 0:
        peak, peak_src = measured_peak()
        alg = B * bytes_per_candidate(J)
        achieved = alg / (kern_ms_max * 1e-3) / 1e9
        dram, ncu_batch = ncu_traffic()
        if dram is not None and ncu_batch:                     # the capture's launch may be a different batch: per candidate
            dram = int(round(dram * B / ncu_batch))
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": dram if headline else None, "eval_path": kernel_path,
                "kernel": "k_eval_tiles<1,%s,true>" % ("true" if ints else "false"),
                "kernel_ms": kern_ms_max, "algorithmic_bytes_per_launch": alg, "peak_source": peak_src,
                "note": "instruction-issue / ALU-pipe bound, not HBM bound: one list-scheduling step is ~51 SASS "
                        "instructions per warp of 32 candidates for 64 bytes of input; see DESIGN.md 5.1 and profiles/"}
        cpu = None
        milp = None
        if world == 1 and not args.no_cpu:
            if milp_proc is not None:
                milp = milp_leg_finish(milp_proc, eng, c4_tasks, solve_leg["makespan"], solve_leg["wall_s"])
            r = cpu_arm(3, 1, args.config if args.config in ("C3", "C4", "C5") else "C4")
            cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"],
                   "ms_per_step_min": r["ms_per_step_min"], "ms_per_step_max": r["ms_per_step_max"]}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_total_max / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": static_config(ints) if headline else {"workload": WORKLOAD, "integer_starts": ints},
                "run": {"candidates_per_gpu_per_step": B,
                        "input_MB_per_gpu_per_step": B * opt.stride(0) * (1 + (1 if J <= 256 else 2)) / 1e6,
                        "exchange": ("none (N=1)" if world == 1 else
                                     ("one MIN of a uint64 per step over NVLink peer memory, fused into the "
                                      "evaluation kernel: publish in the tail, non-blocking fold of the previous "
                                      "step's keys between tiles (last step folded by a one-warp kernel inside the "
                                      "timed region)" if pipelined else
                                      "one MIN of a uint64 per step over NVLink peer memory (publish fused into the "
                                      "evaluation kernel, one-warp fold kernel)") if use_xchg else
                                     "one NCCL all_reduce(MIN) of a uint64 per step"),
                        "start": "host barrier + synchronize, then a device-side rendezvous of all ranks queued in "
                                 "front of the first timed event" if world > 1 else "synchronize",
                        "per_rank": per_rank},
                "clocks": clocks, "e2e": e2e, "solve_api": solve_leg, "search_round": search_leg,
                "gpu_launches": args.steps + (1 if pipelined else 0), "roofline": roof, "cpu_baseline": cpu}
        if milp is not None:
            line["milp"] = milp
        if configs is not None:
            line["configs"] = configs
        if exchange_check is not None:
            line["exchange_check"] = exchange_check
            line["exchange_detail"] = exchange_detail
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
