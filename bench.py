#!/usr/bin/env python
"""bench.py -- vehicle-steps/second of the CityFlow step engine on B200 (BASELINE.json metric).

A "step" is one Engine::nextStep over the whole road network.  Workload at N=1: the 30x30 grid of
BASELINE.json configs[2] with the dense random-walk demand of SURVEY.md Appendix A (frac=0.5, interval=10 s,
~1.3e5 concurrent vehicles).  Both arms first advance the simulation `--prefill` steps (untimed scenario
preparation: the network starts empty) so that the timed steps run at that operating point.

N>1 (`--multi`):
  weak     (default) ONE simulation of a 30 x (30*N) grid cut into N column strips, one strip (~1.3e5 vehicles) per
           GPU, seam records exchanged every step through peer memory over NVLink (device_shard.cuh);
           CITYFLOW_B200_SHARD_TRANSPORT=nccl selects the staged NCCL send/recv form instead
  strong   BASELINE.json configs[3]: the SAME 30x30 grid cut into N strips
  replicas N independent copies of the N=1 workload (no exchange)
`--config rl` measures BASELINE.json configs[4] instead (6x6 grid, rlTrafficLight: per step 36 x set_tl_phase + next_step +
two lane observations), one engine replica per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # our CUDA engine
  python bench.py --impl reference [...]                         # reference CPU engine, host cores (rank 0 only)
  python bench.py [...] --dump-outputs DIR                       # + the last timed step's results as DIR/<name>.npy

Prints ONE JSON line on rank 0 (task contract): value / e2e / roofline / cpu_baseline / clocks / gpu_launches, plus
`parity_check`: the sum of get_vehicle_count() over the timed steps of this run next to the same sum taken from the
compiled reference on the same scenario and the same step window.
"""
import argparse
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "vehicle_steps_per_sec"
UNIT = "vehicle-steps/s"

# The bench grids use a HETEROGENEOUS fleet: every flow's vehicle parameters lie within +-2 % of the generator's
# template.  Reason: the reference orders two vehicles that enter the same lane in the same step with bit-EQUAL distance by
# a non-stable sort over a buffer its worker threads fill in completion order (engine.cpp:247-249, :403-409, :480), so from
# the first such tie on its own result depends on thread timing -- measured: thread_num 3 vs 8, and two runs at 8, give
# different vehicle counts on the 30x60 grid from step 468 on (profiles/r02_reference_ties.md).  With identical vehicles
# such ties occur about once per 3e8 vehicle-steps (1 on 30x30 and on 30x60, 8 on 30x120 before step 1300); with distinct
# parameters none on 30x30 ... 30x240 (oracle tie counter), so parity_check is well defined.  `--fleet-spread 0` gives the
# generator's identical vehicles.
FLEET_SPREAD = 0.02


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=1000)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--config", default="grid", choices=["grid", "rl"], help="grid: BASELINE configs[2]/[3]; rl: configs[4]")
    p.add_argument("--prefill", type=int, default=1200, help="untimed steps that fill the network before timing")
    p.add_argument("--rows", type=int, default=30)
    p.add_argument("--cols", type=int, default=30)
    p.add_argument("--frac", type=float, default=0.5)
    p.add_argument("--flow-interval", type=float, default=10.0)
    p.add_argument("--flow-seed", type=int, default=1)
    p.add_argument("--fleet-spread", type=float, default=-1.0, help="per-flow vehicle parameter spread (default 0.02, see FLEET_SPREAD; 0 = identical vehicles)")
    p.add_argument("--threads", type=int, default=0, help="reference arm: thread_num (default nproc)")
    p.add_argument("--cpu-steps", type=int, default=100, help="cpu_baseline sample: timed steps after the prefill")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-parity", action="store_true", help="skip the reference run behind parity_check")
    p.add_argument("--no-sweep", action="store_true", help="cpu_baseline: thread_num = nproc only, no thread sweep")
    p.add_argument("--lane-change", action="store_true",
                   help='the same workload with "laneChange": true (no parity_check: the reference\'s lane-change schedule '
                        "follows heap addresses, its result is only defined statistically)")
    p.add_argument("--multi", default="weak", choices=["weak", "sharded", "strong", "replicas"],
                   help="N>1, see the module docstring ('sharded' = 'weak')")
    p.add_argument("--clock-ms", type=int, default=50, help="nvidia-smi sampling period (0 = off)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps write what the last of them computed, as a caller of cityflow.Engine receives "
                        "it, to DIR/<name>.npy (float64, at most 64 MB in all): identical arguments give identical inputs, so "
                        "two builds can be compared output for output")
    p.add_argument("--profile-steps", type=int, default=0,
                   help="ncu mode: after prefill+warmup run this many steps between cudaProfilerStart/Stop and exit "
                        "(use with ncu --profile-from-start off)")
    a = p.parse_args()
    if a.multi == "sharded":
        a.multi = "weak"
    if a.lane_change:
        a.no_parity = True
        if a.gpus > 1:
            a.multi = "replicas"   # the lane-change path is single-GPU (its scheduling kernels are not sharded)
    return a


def scenario_module():
    """cityflow_b200/scenario.py loaded by PATH: the reference arm must not import the product package (its __init__
    maps libcityflow_b200.so)."""
    spec = importlib.util.spec_from_file_location("_cfb_scenario", os.path.join(ROOT, "cityflow_b200", "scenario.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def grid_cols(args):
    n = max(args.gpus, 1)
    return args.cols * n if (n > 1 and args.multi == "weak") else args.cols


def flow_seed(args):
    return args.flow_seed


def fleet_spread(args):
    return args.fleet_spread if args.fleet_spread >= 0 else FLEET_SPREAD


def make_scenario(args, directory):
    sc = scenario_module()
    if args.config == "rl":
        return sc.make_grid_scenario(directory, 6, 6, name="rl", rl_traffic_light=True, dense=dict(frac=1.0, interval=5.0, seed=2))
    return sc.make_grid_scenario(directory, args.rows, grid_cols(args), name="bench", lane_change=args.lane_change,
                                 dense=dict(frac=args.frac, interval=args.flow_interval, seed=flow_seed(args), fleet_spread=fleet_spread(args)))


def workload_name(args):
    if args.config == "rl":
        return "RL loop: 6x6 grid, rlTrafficLight, random-walk flows frac=1 interval=5s seed=2; per step 36 x set_tl_phase + next_step + get_lane_vehicle_count + get_lane_waiting_vehicle_count"
    fs = fleet_spread(args)
    return "%dx%d grid (tools/generator layout), random-walk flows frac=%g interval=%gs seed=%d%s, interval=1.0s, seed=0" % (
        args.rows, grid_cols(args), args.frac, args.flow_interval, flow_seed(args),
        (", vehicle parameters per flow within +-%g%% of the template" % (100 * fs)) if fs > 0 else "") + (
        ", laneChange=true" if args.lane_change else "")


def scaling_of(args):
    return "strong" if (args.gpus > 1 and args.multi == "strong") else "weak"


# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons (B200_PROFILING.md recipe).  Runs for the whole life of the process;
    mark() remembers how many samples exist at a moment, so a window of the log can be summarised afterwards."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device=0, period_ms=50):
        self.device, self.period_ms, self.proc, self.path = device, period_ms, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile(prefix="clocks_", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def mark(self):
        try:
            with open(self.path) as f:
                return sum(1 for _ in f)
        except Exception:
            return 0

    def stop(self, lo=0, hi=None, lo_fallback=0):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        time.sleep(max(self.period_ms, 20) / 1e3)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = []
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    rows.append((float(c[1]), float(c[2]), [n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]) if v.lower().startswith("active")]))
                except ValueError:
                    continue
            os.unlink(self.path)
        except Exception:
            pass
        window, what = rows[lo:hi], "timed region (value, value_l2_warm, e2e)"
        if len(window) < 2:   # the timed region is shorter than a sampling period or two: include the GPU work before it
            window, what = rows[lo_fallback:hi], "prefill + warm-up + timed region (the timed region alone is shorter than two sampling periods)"
        if window:
            out.update(sm_mhz=statistics.median(r[0] for r in window), sm_max_mhz=max(r[1] for r in window),
                       reasons=sorted({n for r in window for n in r[2]}), samples=len(window), window=what, period_ms=self.period_ms)
        return out


def measured_peak_gbs():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json, copy bandwidth)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md, 6.65 TB/s)"


# ----------------------------------------------------------------------------------------------
# Reference side (oracle/ is test infrastructure: only this leg of bench.py runs it, always as a subprocess)
def reference_run(cfg, steps, warmup_total, threads, want_counts=False):
    """The reference's own CPU engine (unmodified sources compiled into oracle/_ref) or, when that build did not
    travel, the CPU restatement (single thread).  Returns throughput and, on request, get_vehicle_count() after
    every step (warm-up included)."""
    from oracle import harness as H
    if H.have_ref():
        path = tempfile.mktemp(suffix=".bin") if want_counts else None
        cmd = [H.REFDUMP, "bench", cfg, str(steps), str(threads), str(warmup_total)] + ([path] if path else [])
        out = subprocess.check_output(cmd, timeout=3600)
        r = json.loads(out.decode().strip().splitlines()[-1])
        counts = None
        if path:
            import numpy as np
            counts = np.fromfile(path, "<i4").astype("int64")
            os.unlink(path)
        return dict(kind="reference", cores=threads, value=r["vehicle_steps_per_s"], seconds=r["seconds"],
                    vehicle_steps=r["vehicle_steps"], final_vehicles=r["final_vehicles"], counts=counts)
    if not H.have_port():
        H.build(ref=False)
    import numpy as np
    o = H.PortOracle(cfg)
    counts = []
    for _ in range(warmup_total):
        o.next_step()
        counts.append(o.vehicle_count())
    vs = 0
    t0 = time.perf_counter()
    for _ in range(steps):
        o.next_step()
        counts.append(o.vehicle_count())
        vs += counts[-1]
    sec = time.perf_counter() - t0
    return dict(kind="port", cores=1, value=vs / sec, seconds=sec, vehicle_steps=vs, final_vehicles=o.vehicle_count(),
                counts=np.array(counts, "int64"))


def reference_sweep(cfg, steps, warmup_total, nproc):
    """BASELINE.md section 3.2: thread_num swept at one operating point (state handed over through the reference's own
    Archive), headline denominator thread_num = nproc, best-of-sweep as the stricter one."""
    from oracle import harness as H
    if not H.have_ref():
        return None
    ts = [nproc] + [t for t in (8, 16, 32, 64) if t < nproc]
    out = subprocess.check_output([H.REFDUMP, "sweep", cfg, str(steps), str(warmup_total), ",".join(str(t) for t in ts)], timeout=3600)
    r = json.loads(out.decode().strip().splitlines()[-1])
    table = {int(t): v["vehicle_steps_per_s"] for t, v in r["sweep"].items()}
    best = max(table, key=table.get)
    return {"table": table, "best_threads": best, "best_value": table[best], "nproc_value": table[nproc],
            "mean_vehicles": r["sweep"][str(nproc)]["vehicle_steps"] / max(steps, 1)}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.config == "rl":
        return run_reference_rl(args)
    nproc = os.cpu_count() or 1
    threads = args.threads or nproc
    with tempfile.TemporaryDirectory() as d:
        cfg = make_scenario(args, d)
        r = reference_run(cfg, args.steps, args.prefill + args.warmup, threads)
        sweep = None
        if not args.no_sweep and r["kind"] == "reference" and args.gpus <= 1:   # (one operating point: the N=1 workload)
            try:
                sweep = reference_sweep(cfg, min(args.steps, 50), args.prefill + args.warmup, nproc)
            except Exception as ex:  # noqa: BLE001
                sweep = {"error": repr(ex)}
    sample = "%d timed steps after %d untimed steps, thread_num=%d" % (args.steps, args.prefill + args.warmup, r["cores"])
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"] / max(args.steps, 1),
        "higher_is_better": True, "scaling": scaling_of(args), "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args), "prefill_steps": args.prefill,
                   "mean_vehicles": r["vehicle_steps"] / max(args.steps, 1), "host_cores": nproc,
                   "note": "reference CPU engine runs once on rank 0 regardless of --gpus"},
        "vehicle_steps_in_timed_window": r["vehicle_steps"],
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": sample,
                         "thread_sweep": sweep},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


DUMP_VEHICLES_MAX = 1 << 21   # vehicle arrays above this length are dumped as a fixed, seeded sample (2 x 16 MB)


def write_outputs(directory, arrays):
    """--dump-outputs: one float64 DIR/<name>.npy per array."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def engine_outputs(eng, ranks, sharded):
    """The results of the step just taken as a caller of cityflow.Engine receives them: the vehicle count, per-lane vehicle
    and waiting counts in lane_ids() order, and every running vehicle's speed and distance in the order of its id (all
    ranks of a sharded run call this: the lane getters are collective, each rank reports the vehicles of its strip)."""
    import numpy as np
    out = {"vehicle_count": eng.get_vehicle_count()}
    lanes = eng.lane_ids()
    cnt, wait = eng.get_lane_vehicle_count(), eng.get_lane_waiting_vehicle_count()
    out["lane_vehicle_count"] = [cnt[k] for k in lanes]
    out["lane_waiting_vehicle_count"] = [wait[k] for k in lanes]
    speed, distance = eng.get_vehicle_speed(), eng.get_vehicle_distance()
    if sharded:
        parts = [None] * ranks.world if ranks.rank == 0 else None
        ranks.dist.gather_object((speed, distance), parts, dst=0)
        if ranks.rank != 0:
            return None
        speed, distance = {}, {}
        for sp, di in parts:
            speed.update(sp)
            distance.update(di)
    ids = sorted(speed)
    pick = np.arange(len(ids))
    if len(ids) > DUMP_VEHICLES_MAX:
        pick = np.sort(np.random.default_rng(0).choice(len(ids), DUMP_VEHICLES_MAX, replace=False))
        out["vehicle_sample_index"] = pick
    out["vehicle_speed"] = [speed[ids[i]] for i in pick]
    out["vehicle_distance"] = [distance[ids[i]] for i in pick]
    return out


# ----------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local)
    sampler = ClockSampler(local, args.clock_ms)
    if int(os.environ.get("RANK", "0")) == 0 and args.clock_ms > 0:
        sampler.start()
    from cityflow_b200.distutil import Ranks
    ranks = Ranks("nccl", torch.device("cuda", local))
    world, rank, dist = ranks.world, ranks.rank, ranks.dist
    if args.config == "rl":
        return run_ours_rl(args, ranks, sampler)

    import cityflow  # our drop-in module (repo root)
    import cityflow_b200
    sharded = world > 1 and args.multi in ("weak", "strong")
    tmp = tempfile.TemporaryDirectory()
    cfg = make_scenario(args, tmp.name)
    t0 = time.perf_counter()
    if sharded:
        ids = [cityflow_b200.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        eng = cityflow.Engine(cfg, thread_num=1, device=local, shard_rank=rank, shard_world=world, nccl_id=ids[0])
    else:
        eng = cityflow.Engine(cfg, thread_num=1, device=local)
    load_s = time.perf_counter() - t0

    def barrier():
        ranks.barrier()
        torch.cuda.synchronize()
        eng.synchronize()

    reduce_max, reduce_sum = ranks.max, ranks.sum

    # ---- scenario preparation + warm-up ----
    m_prefill = sampler.mark() if rank == 0 else 0
    eng.next_steps(args.prefill)
    eng.synchronize()
    warm = max(args.warmup, 3)
    eng.timed_steps(warm, True)
    n_start = eng.get_vehicle_count()
    if args.profile_steps > 0:  # profiling run: numbers printed under a profiler are never bench values
        cudart = torch.cuda.cudart()
        cudart.cudaProfilerStart()
        eng.timed_steps(args.profile_steps, True)
        cudart.cudaProfilerStop()
        if rank == 0:
            sampler.stop()
            print(json.dumps({"profiled_steps": args.profile_steps, "vehicles": n_start}))
        return

    # ---- value: K steps, device time (CUDA events on the engine stream), L2 flushed between steps ----
    barrier()
    m_lo = sampler.mark() if rank == 0 else 0
    launches0 = eng.gpu_launches()
    ms_flush, vs_flush = eng.timed_steps(args.steps, True)
    barrier()
    launches = eng.gpu_launches() - launches0
    ties_window = reduce_sum(eng.tie_count())
    ms_flush_max = reduce_max(ms_flush)
    vs_total = reduce_sum(vs_flush)
    value = vs_total / (ms_flush_max / 1e3)

    # same, back to back without flush (state stays L2 resident, as in real stepping); median of chunks so that one
    # host hiccup (the host paces this loop) does not decide the number
    chunks = []
    barrier()
    left = args.steps
    while left > 0:
        k = min(left, max(10, args.steps // 8))
        ms_w, vs_w = eng.timed_steps(k, False)
        chunks.append((reduce_max(ms_w) / k, reduce_sum(vs_w) / k))
        left -= k
    barrier()
    ms_warm_step = statistics.median(c[0] for c in chunks)
    value_warm = statistics.mean(c[1] for c in chunks) / (ms_warm_step / 1e3)

    # ---- e2e: the user-visible loop through the public API, host clock, H2D + D2H every step ----
    h2d0, d2h0 = eng.transfer_bytes()
    barrier()
    t0 = time.perf_counter()
    acc = 0
    for _ in range(args.steps):
        eng.next_step()
        acc += eng.get_vehicle_count()
    e2e_s = time.perf_counter() - t0
    barrier()
    m_hi = sampler.mark() if rank == 0 else 0
    if args.dump_outputs:   # the last timed step: the end of the e2e loop (the kernel-timing pass below is untimed)
        outputs = engine_outputs(eng, ranks, sharded)
        if rank == 0:
            write_outputs(args.dump_outputs, outputs)
    h2d1, d2h1 = eng.transfer_bytes()
    host_gen_ms, host_enq_ms = eng.host_times()
    # sharded: get_vehicle_count() already is the network-wide count on every rank
    e2e_value = (acc if sharded else reduce_sum(acc)) / reduce_max(e2e_s)
    clocks = sampler.stop(m_lo, m_hi, m_prefill) if rank == 0 else {}

    eng_steps_total = args.prefill + warm + 3 * args.steps
    # ---- per-kernel device time (CUDA events around every kernel; separate pass, serialised) ----
    shard_phases = None
    if sharded:   # phase by phase (CUDA events between the phases; plain launches, serialised): where a sharded step's time goes
        (k_ing, k_not, k_ctl, k_mov, k_led), kn = (0.0, 0.0, 0.0, 0.0, 0.0), 1
        eng.enable_kernel_timing(True)
        for _ in range(min(args.steps, 50)):
            eng.next_step()
        ph, pn = eng.shard_phase_times()
        eng.enable_kernel_timing(False)
        names = ["k_ingest", "k_notify+k_control", "send_movers", "recv_movers(+wait)", "k_move", "send_tails", "recv_tails(+wait)", "k_leader"]
        shard_phases = {"rank0_ms": {n: v / max(pn, 1) for n, v in zip(names, ph)},
                        "max_over_ranks_ms": {n: reduce_max(v / max(pn, 1)) for n, v in zip(names, ph)}}
    else:
        eng.enable_kernel_timing(True)
        ksteps = min(args.steps, 50)
        for _ in range(ksteps):
            eng.next_step()
        (k_ing, k_not, k_ctl, k_mov, k_led), kn = eng.kernel_times()
        kn = max(kn, 1)   # (a lane-change step is not the five-kernel sequence: no per-kernel times)
        eng.enable_kernel_timing(False)
    n_now = eng.get_vehicle_count()
    n_drv = eng.num_drivables() if hasattr(eng, "num_drivables") else 0
    kms = {"k_ingest": k_ing / kn, "k_notify": k_not / kn, "k_control": k_ctl / kn, "k_move": k_mov / kn, "k_leader": k_led / kn}
    dominant = max(kms, key=kms.get)
    peak, peak_src = measured_peak_gbs()
    # algorithmic bytes per launch (DESIGN.md section 5): per running vehicle N, per drivable D
    # The leader scan (SURVEY.md 8d: 32 B per vehicle + 12 B per drivable) no longer has a kernel of its own: k_move settles
    # leader / gap of every non-head while it holds the bucket in registers (its reads are k_move's own; it adds the 12 B
    # written per vehicle), k_leader is left with the list heads (one per occupied drivable).
    alg = {
        "k_leader": 12 * n_drv + 64 * min(n_drv, n_now),   # per occupied drivable: head record (kin, ids, nav = 48) + tail gather 16
        "k_control": 96 * n_now + 4 * n_drv,
        "k_move": (88 + 12) * n_now + 8 * n_drv,           # commit (88 B) + the leader scan's writes (leader 4 + gap 8)
        "k_notify": 16 * n_now + 24 * (n_drv),
        "k_ingest": 12 * n_drv,
    }
    try:  # DRAM bytes per launch from the committed ncu --set full capture (same workload)
        traffic = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic_bytes_per_launch.json")))
    except Exception:
        traffic = {}
    same_workload = (args.rows, args.cols, args.frac, args.flow_interval) == (30, 30, 0.5, 10.0)

    def roof(k):
        gbs = alg[k] / (kms[k] * 1e-3) / 1e9 if kms[k] > 0 else 0.0
        return {"kernel": k, "bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                "traffic": traffic.get(k) if same_workload else None,
                "note": "latency-bound at this size (state is L2-sized; dependent loads + FP64 div/sqrt chains), see profiles/",
                "algorithmic_bytes_per_launch": alg[k], "avg_launch_ms": kms[k], "peak_source": peak_src}

    line = None
    if rank == 0:
        mean_n = vs_total / max(args.steps, 1)
        if sharded:
            par = ("%s scaling: %d column strips of ONE simulation; seam records (entrants, tail records, blocker changes) %s"
                   % (scaling_of(args), world, "stored into the neighbours' mailboxes through peer memory (NVLink), 2 dependent hops per step, no collective"
                      if os.environ.get("CITYFLOW_B200_SHARD_TRANSPORT", "") != "nccl" else "staged and moved by 2 NCCL send/recv groups per step"))
        else:
            par = "replicas x%d (one engine per GPU, no exchange)" % world
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms_flush_max / max(args.steps, 1), "higher_is_better": True, "scaling": scaling_of(args),
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": workload_name(args), "prefill_steps": args.prefill, "mean_vehicles": mean_n,
                "mean_vehicles_per_gpu": mean_n / world, "vehicles_at_start": n_start, "parallelism": par,
                "l2": "value: 256 MiB memset between timed steps (state ~30 MB would otherwise stay L2-resident); "
                      "value_l2_warm and e2e: steps back to back as in real stepping",
                "load_seconds": load_s,
            },
            "value_l2_warm": value_warm,
            "ms_per_step_l2_warm": ms_warm_step,
            "e2e": {"value": e2e_value, "unit": UNIT,
                    "h2d_bytes_per_step": (h2d1 - h2d0) / max(args.steps, 1),
                    "d2h_bytes_per_step": (d2h1 - d2h0) / max(args.steps, 1),
                    "ms_per_step": 1e3 * e2e_s / max(args.steps, 1),
                    "api": "cityflow.Engine.next_step() + get_vehicle_count() every step"},
            "gpu_launches": int(launches),
            "kernel_ms": kms,
            "host_ms_per_step": {"spawn_generation": host_gen_ms / max(eng_steps_total, 1), "enqueue": host_enq_ms / max(eng_steps_total, 1)},
            "shard_phase_ms": shard_phases,
            "roofline": roof(dominant) if not sharded else None,
            "roofline_leader_scan": dict(roof("k_move"), note="the leader scan is fused into k_move (non-heads: shuffle over the "
                                         "registers that compact the bucket); list heads: k_leader, %.4f ms" % kms["k_leader"]) if not sharded else None,
            "clocks": clocks,
        }
    if dist is not None:
        dist.barrier()
    # ---- reference on this box's host cores (rank 0): parity of the timed window (every N) + cpu_baseline (N=1) ----
    if rank == 0 and not (args.no_parity and (args.no_cpu_baseline or world > 1)):
        nproc = os.cpu_count() or 1
        threads = args.threads or nproc
        first = args.prefill + warm            # steps before the `value` window
        try:
            ref_steps = max(args.steps, args.cpu_steps) if (world == 1 and not args.no_cpu_baseline) else args.steps
            r = reference_run(cfg, ref_steps, first, threads, want_counts=not args.no_parity)
            if not args.no_parity:
                ref_vs = int(r["counts"][first:first + args.steps].sum())
                line["parity_check"] = {
                    "ours_vehicle_steps": int(vs_total), "reference_vehicle_steps": ref_vs, "equal": int(vs_total) == ref_vs,
                    "window": "steps %d..%d" % (first + 1, first + args.steps),
                    "ties_reference_order_undefined": int(ties_window),
                    "what": "sum of get_vehicle_count() after each timed step: this engine (all ranks) vs oracle/_ref (unmodified "
                            "reference, thread_num=%d) on the same scenario" % r["cores"]}
            if world == 1 and not args.no_cpu_baseline:
                cb = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                      "sample": "%d timed steps after %d untimed steps of the same scenario (mean %.0f vehicles)" % (
                          ref_steps, first, r["vehicle_steps"] / max(ref_steps, 1))}
                if not args.no_sweep and r["kind"] == "reference":
                    try:
                        sw = reference_sweep(cfg, min(args.cpu_steps, 50), first, nproc)
                        cb["thread_sweep"] = sw
                        cb["best_of_sweep"] = {"value": sw["best_value"], "cores": sw["best_threads"]}
                    except Exception as ex:  # noqa: BLE001
                        cb["thread_sweep"] = {"error": repr(ex)}
                line["cpu_baseline"] = cb
        except Exception as ex:  # keep the GPU numbers even if the CPU arm fails
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": threads, "kind": "reference", "sample": "failed: %r" % (ex,)}
    if rank == 0:
        print(json.dumps(line))
    del eng
    tmp.cleanup()
    ranks.close()


# ----------------------------------------------------------------------------------------------
# BASELINE.json configs[4]: the RL inner loop, one independent engine replica per GPU ("replicas only": no exchange)
def rl_loop(mod, cfg, inters, steps, threads=1, keep=None, **kw):
    eng = mod.Engine(cfg, thread_num=threads, **kw)
    if keep is not None:
        keep.append(eng)   # the reference's ~Engine can hang with worker threads parked on its barriers: the caller exits without it
    for _ in range(100):
        eng.next_step()
    vs = 0
    t0 = time.perf_counter()
    for t in range(steps):
        ph = (t // 30) % 8
        for i in inters:
            eng.set_tl_phase(i, ph)
        eng.next_step()
        c = eng.get_lane_vehicle_count()
        w = eng.get_lane_waiting_vehicle_count()
        vs += eng.get_vehicle_count()
    sec = time.perf_counter() - t0
    return {"seconds": sec, "vehicle_steps": vs, "lanes": len(c), "waiting_last": sum(w.values())}


def rl_intersections(cfg):
    net = json.load(open(os.path.join(os.path.dirname(cfg), "roadnet_rl.json")))
    return [i["id"] for i in net["intersections"] if not i["virtual"]]


def run_ours_rl(args, ranks, sampler):
    import torch
    import cityflow
    import cityflow_b200
    world, rank = ranks.world, ranks.rank
    local = int(os.environ.get("LOCAL_RANK", "0"))
    tmp = tempfile.TemporaryDirectory()
    cfg = make_scenario(args, tmp.name)
    inters = rl_intersections(cfg)
    ranks.barrier()
    m_lo = sampler.mark() if rank == 0 else 0
    r = rl_loop(cityflow, cfg, inters, args.steps, device=local)
    # the same loop with observations / actions staying on the GPU (cityflow_b200 extras; a stand-in policy of a few torch ops)
    eng = cityflow.Engine(cfg, thread_num=1, device=local)
    for _ in range(100):
        eng.next_step()
    n_int = eng.num_intersections()
    obs = cityflow_b200.LaneObservations(eng)
    cnt, wait = obs.vehicle_count, obs.waiting_count
    n_lanes = len(obs.lane_ids)
    key = (torch.arange(n_lanes, device=cnt.device) * n_int // n_lanes).to(torch.int64) * 8 + (torch.arange(n_lanes, device=cnt.device) % 8).to(torch.int64)
    votes = torch.zeros(n_int * 8, device=cnt.device, dtype=torch.int32)
    vs_dev = torch.zeros((), device=cnt.device, dtype=torch.int64)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        obs.refresh()
        votes.zero_()
        votes.index_add_(0, key, wait)
        cityflow_b200.set_tl_phases_tensor(eng, votes.view(n_int, 8).argmax(1).to(torch.int32))
        eng.next_step()
        vs_dev += cnt.sum()
    torch.cuda.synchronize()
    eng.synchronize()
    dev_s = time.perf_counter() - t0
    if args.dump_outputs and rank == 0:   # the last timed step of the device-resident loop: its actions and what it left
        actions = votes.view(n_int, 8).argmax(1)
        obs.refresh()
        write_outputs(args.dump_outputs, {"tl_phases": actions.cpu(), "lane_vehicle_count": cnt.cpu(), "lane_waiting_vehicle_count": wait.cpu(),
                                          "lane_speed_sum": obs.speed_sum.cpu(), "vehicle_steps": int(vs_dev)})
    ranks.barrier()
    m_hi = sampler.mark() if rank == 0 else 0
    sec = ranks.max(r["seconds"])
    vs = ranks.sum(r["vehicle_steps"])
    dsec, dvs = ranks.max(dev_s), ranks.sum(int(vs_dev))
    if rank == 0:
        clocks = sampler.stop(m_lo, m_hi, 0)
        n_l = r["lanes"]
        line = {
            "metric": METRIC, "value": vs / sec, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": 100,
            "ms_per_step": 1e3 * sec / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload_name(args), "parallelism": "replicas x%d (one engine per GPU, no exchange)" % world,
                       "mean_vehicles_per_replica": vs / args.steps / world},
            "env_steps_per_s": world * args.steps / sec,
            "e2e": {"value": vs / sec, "unit": UNIT, "h2d_bytes_per_step": 4 * len(inters) + 64, "d2h_bytes_per_step": 8 * n_l + 64,
                    "api": "36 x set_tl_phase + next_step + get_lane_vehicle_count + get_lane_waiting_vehicle_count + get_vehicle_count (Python dicts)"},
            "device_resident_api": {"env_steps_per_s": world * args.steps / dsec, "vehicle_steps_per_s": dvs / dsec,
                                    "api": "LaneObservations.refresh + torch policy + set_tl_phases_tensor + next_step, no host copies"},
            "gpu_launches": None, "clocks": clocks,
        }
        print(json.dumps(line))
    ranks.close()


def run_reference_rl(args):
    """BASELINE.md section 3.5: N reference processes with thread_num=1 (one per GPU replica) and one with thread_num=nproc."""
    code = ("import sys, json; sys.path.insert(0, %r); import bench; from oracle import harness as H; m = H.load_reference_module();"
            "import os; keep = []; r = bench.rl_loop(m, sys.argv[1], json.loads(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4]), keep); print(json.dumps(r));"
            "sys.stdout.flush(); os._exit(0)" % ROOT)
    n = max(args.gpus, 1)
    nproc = os.cpu_count() or 1
    with tempfile.TemporaryDirectory() as d:
        cfg = make_scenario(args, d)
        inters = json.dumps(rl_intersections(cfg))
        t0 = time.perf_counter()
        procs = [subprocess.Popen([sys.executable, "-c", code, cfg, inters, str(args.steps), "1"], stdout=subprocess.PIPE) for _ in range(n)]
        outs = [json.loads(p.communicate()[0].decode().strip().splitlines()[-1]) for p in procs]
        _ = time.perf_counter() - t0
        big = json.loads(subprocess.check_output([sys.executable, "-c", code, cfg, inters, str(args.steps), str(nproc)]).decode().strip().splitlines()[-1])
    sec = max(o["seconds"] for o in outs)
    vs = sum(o["vehicle_steps"] for o in outs)
    line = {
        "impl": "reference", "metric": METRIC, "value": vs / sec, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": 100,
        "ms_per_step": 1e3 * sec / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args), "parallelism": "%d reference processes, thread_num=1 each" % n, "host_cores": nproc},
        "env_steps_per_s": n * args.steps / sec,
        "one_process_thread_num_nproc": {"env_steps_per_s": args.steps / big["seconds"], "vehicle_steps_per_s": big["vehicle_steps"] / big["seconds"], "threads": nproc},
        "cpu_baseline": {"value": vs / sec, "unit": UNIT, "cores": n, "kind": "reference", "sample": "%d env steps per process after 100 untimed" % args.steps},
        "e2e": {"value": vs / sec, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
