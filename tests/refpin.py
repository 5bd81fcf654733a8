"""Results of the UNMODIFIED reference, pinned in tests/golden/reference/ so that the comparisons with it run anywhere.

The tests that compare with the reference used to run it live (oracle/_ref, compiled from the reference's sources).  They
now compare with what it computed, recorded once by this module on the same seeded scenarios:

    make -C oracle ref REF=<reference source tree>
    python tests/refpin.py [name ...]

A state is pinned as one 64-bit digest per part (vehicle count, per-lane arrays, every running vehicle's fields, list
order, ...) over a group of consecutive compared states, so "equal in every compared field at every compared step" is
kept while the fixtures stay small: {"parts", "group", "steps": [[first, last] per group], "digests": {part: "<one hex
digest per group, space-separated>"}}.  Each part is hashed from the same normalised bytes on both sides: vehicles sorted
by (flow, index) -- lane-change records in priority order, as dumped -- integers as little-endian int32 / int64,
doubles as their IEEE-754 bits with -0.0 folded into +0.0 (the comparisons treat them as equal)."""
import gzip
import hashlib
import json
import os
import struct
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PINS = os.path.join(HERE, "golden", "reference")
if ROOT not in sys.path:
    sys.path.append(ROOT)          # appended: a child process's `import cityflow` stays whatever its PYTHONPATH puts first
from oracle import harness as H   # noqa: E402

# harness.compare_states: exact fields of every running vehicle
VEH_INT = ("flow", "cnt", "priority", "drivable", "leader_flow", "leader_cnt", "blocker_flow", "blocker_cnt")
VEH_FLOAT = ("dis", "speed", "gap")
# tests/archive_checks.py STATE_FIELDS (no enterLaneLinkTime)
STATE_INT = ("flow", "cnt", "priority", "drivable", "leader_flow", "leader_cnt", "blocker_flow", "blocker_cnt")

FULL = ("vehicle_count", "totals", "lane_count", "lane_waiting", "lane_queue", "phases", "vehicles")
GPU = ("vehicle_count", "lane_count", "lane_waiting", "vehicles")
LC = ("vehicle_count", "totals", "lane_count", "phases", "lc_vehicles", "order")


def _i4(a):
    return np.ascontiguousarray(a, dtype="<i4").tobytes()


def _f8(a):
    a = np.array(a, dtype="<f8")
    a[a == 0] = 0.0
    return a.tobytes()


def part_bytes(st, part):
    if part == "vehicle_count":
        return struct.pack("<q", int(st.vehicle_count))
    if part == "totals":
        return struct.pack("<qq", int(st.pool_size), int(st.finished)) + _f8([st.cum_travel_time])
    if part in ("lane_count", "lane_waiting", "lane_queue", "phases"):
        return _i4(getattr(st, part))
    if part in ("vehicles", "state"):
        v = st.key_sorted()
        b = [_i4(v[f]) for f in (VEH_INT if part == "vehicles" else STATE_INT)] + [_f8(v[f]) for f in VEH_FLOAT]
        if part == "vehicles":
            b.append(np.ascontiguousarray(v["enter_ll_time"], dtype="<i8").tobytes())
        return b"".join(b)
    if part == "lc_vehicles":
        v = st.vehicles
        return b"".join(_f8(v[f]) if v.dtype[f].kind == "f" else _i4(v[f]) for f in H.LC_DTYPE.names)
    if part == "order":
        return b"".join(_i4([o.size]) + _i4(np.ravel(o)) for o in st.order)
    raise KeyError(part)


def digest(data: bytes) -> str:
    return hashlib.sha256(data).hexdigest()[:16]


def lane_digest(a) -> str:
    """digest of a per-lane int array (lane index order)"""
    return digest(_i4(a))


def canonical(x):
    """JSON-like value -> text that is equal exactly when the values are equal (numbers as the bits of a double)."""
    def c(y):
        if isinstance(y, dict):
            return {str(k): c(v) for k, v in y.items()}
        if isinstance(y, (list, tuple)):
            return [c(v) for v in y]
        if isinstance(y, (bool, str)) or y is None:
            return y
        if isinstance(y, (int, float, np.integer, np.floating)):
            return float(y).hex() if float(y) != 0 else "0"
        raise TypeError(type(y))
    return json.dumps(c(x), sort_keys=True)


def value_digest(x) -> str:
    return digest(canonical(x).encode())


class Trail:
    """Digests of a run's states, part by part, `group` states per entry."""

    def __init__(self, parts, group=1):
        self.parts, self.group = tuple(parts), group
        self.entries, self._h, self._n, self._first = [], None, 0, None

    def add(self, step, st):
        if self._h is None:
            self._h, self._first = {p: hashlib.sha256() for p in self.parts}, step
        for p in self.parts:
            self._h[p].update(part_bytes(st, p))
        self._n += 1
        if self._n == self.group:
            return self.close(step)
        return None

    def close(self, step):
        if self._h is None:
            return None
        e = {"steps": [self._first, step]}
        e.update({p: h.hexdigest()[:16] for p, h in self._h.items()})
        self.entries.append(e)
        self._h, self._n = None, 0
        return e


    def pin(self):
        """the pinned form of the entries"""
        return {"parts": list(self.parts), "group": self.group, "steps": [e["steps"] for e in self.entries],
                "digests": {p: " ".join(e[p] for e in self.entries) for p in self.parts}}


class Follow(Trail):
    """A Trail checked entry by entry against a pinned one (`parts`: those this side can produce)."""

    def __init__(self, pin, parts=None, tag=""):
        super().__init__(parts or pin["parts"], pin["group"])
        self.want, self.tag = [{"steps": st} for st in pin["steps"]], tag
        assert set(self.parts) <= set(pin["parts"]), (self.parts, pin["parts"])
        for p in self.parts:
            for w, d in zip(self.want, pin["digests"][p].split()):
                w[p] = d

    def close(self, step):
        e = super().close(step)
        if e is not None:
            k = len(self.entries) - 1
            assert k < len(self.want), "%s: more states than the reference run" % self.tag
            w = self.want[k]
            assert e["steps"] == w["steps"], (self.tag, e["steps"], w["steps"])
            bad = [p for p in self.parts if e[p] != w[p]]
            assert not bad, "%s steps %d..%d: %s differ from the reference" % (self.tag, w["steps"][0], w["steps"][1], ", ".join(bad))
        return e

    def finish(self, step=None):
        if step is not None:
            self.close(step)
        assert len(self.entries) == len(self.want), "%s: %d of %d reference states compared" % (self.tag, len(self.entries), len(self.want))


def load(name):
    with open(os.path.join(PINS, name + ".json")) as f:
        return json.load(f)


def blob(name) -> bytes:
    with gzip.open(os.path.join(PINS, name + ".gz")) as f:
        return f.read()


def static_digests(lane_length, link_length, crosses, n_cross):
    cr = b"".join(struct.pack("<iii", int(c[0]), int(c[1]), int(c[2])) + _f8([c[3], c[4]]) for c in crosses)
    return {"n_lanes": len(lane_length), "n_links": len(link_length), "n_cross": int(n_cross),
            "lane_length": digest(_f8(lane_length)), "link_length": digest(_f8(link_length)), "crosses": digest(cr)}


def ref_static(cfg):
    s = H.RefDump.static(cfg)
    return static_digests([l["length"] for l in s["lanes"]], [l["length"] for l in s["links"]],
                          [c for l in s["links"] for c in l["crosses"]], s["n_cross"])


def python_api_run(ora, cfg, steps, ref=None):
    """The script of tests/test_cpu.py::test_port_oracle_vs_reference_python_api: set_tl_phase, push_vehicle,
    set_vehicle_speed, set_vehicle_route, set_random_seed and reset, applied to the restatement (and, when recording,
    identically to the reference's own Python module).  Yields (step, observations of the engine under test, counters)
    after every step; with `ref` the observations are the reference's and are first asserted equal to the restatement's."""
    c = json.load(open(cfg))
    net = json.load(open(c["dir"] + c["roadnetFile"]))
    inter_ids = [i["id"] for i in net["intersections"]]
    real = [k for k, i in enumerate(net["intersections"]) if not i["virtual"]]
    lane_ids = ["%s_%d" % (r["id"], k) for r in net["roads"] for k in range(len(r["lanes"]))]
    flows = json.load(open(c["dir"] + c["flowFile"]))
    some_route = flows[3]["route"]
    stats = dict(leaders=0, custom=0, rerouted_ok=0, rerouted_no=0)

    def vid(flow, cnt):
        return "manually_pushed_%d" % cnt if flow == -2 else "flow_%d_%d" % (flow, cnt)

    def observe_restatement(v, sample):
        leaders = []
        for f, k in sample:
            lead = ora.get_leader(int(f), int(k))
            leaders.append("" if lead is None else vid(*lead))
        return {"count": ora.vehicle_count(), "time": ora.lib.cfo_current_time(ora.h),
                "lanes": ora.lane_vehicle_count().tolist(), "waiting": ora.lane_waiting_count().tolist(),
                "speed": {vid(f, k): s for f, k, s in zip(v["flow"], v["cnt"], v["speed"])},
                "distance": {vid(f, k): s for f, k, s in zip(v["flow"], v["cnt"], v["dis"])},
                "travel_time": ora.average_travel_time(), "leaders": leaders}

    def observe_reference(sample):
        cnt, wait = ref.get_lane_vehicle_count(), ref.get_lane_waiting_vehicle_count()
        return {"count": ref.get_vehicle_count(), "time": ref.get_current_time(),
                "lanes": [cnt[x] for x in lane_ids], "waiting": [wait[x] for x in lane_ids],
                "speed": ref.get_vehicle_speed(), "distance": ref.get_vehicle_distance(),
                "travel_time": ref.get_average_travel_time(), "leaders": [ref.get_leader(vid(f, k)) for f, k in sample]}

    for s in range(1, steps + 1):
        rerouted = []
        if s % 10 == 1:                      # RL actions
            for k in real:
                ph = (s // 10 + k) % 8
                if ref is not None:
                    ref.set_tl_phase(inter_ids[k], ph)
                ora.set_tl_phase(k, ph)
        if s in (40, 41, 150):               # draws from the engine RNG
            info = {"speed": 3.0, "length": 6.5, "maxSpeed": 12.0} if s != 41 else {}
            if ref is not None:
                ref.push_vehicle(info, some_route)
            ora.push_vehicle(info, some_route)
        if s == 260:
            if ref is not None:
                ref.set_random_seed(77)
            ora.set_random_seed(77)
        if s in (330, 420):
            if ref is not None:
                ref.reset(seed=(s == 420))
            ora.reset(seed=(s == 420))
        if s % 25 == 3:
            v = ora.vehicles()
            for j in range(0, len(v), max(1, len(v) // 5)):
                f, k, sp = int(v["flow"][j]), int(v["cnt"][j]), float(v["speed"][j]) * 0.5
                if ref is not None:
                    ref.set_vehicle_speed(vid(f, k), sp)
                assert ora.set_vehicle_speed(f, k, sp)
                stats["custom"] += 1
        if s % 30 == 7:                      # re-route vehicles that are under way
            v = ora.vehicles()
            for j in range(1, len(v), max(1, len(v) // 9)):
                f, k = int(v["flow"][j]), int(v["cnt"][j])
                target = flows[(s + j) % len(flows)]["route"][-1:] if j % 3 else ["no_such_road"]
                b = ora.set_vehicle_route(f, k, target)
                if ref is not None:
                    a = ref.set_vehicle_route(vid(f, k), target)
                    assert a == b, (s, vid(f, k), target, a, b)
                rerouted.append(b)
                stats["rerouted_ok" if b else "rerouted_no"] += 1
        if ref is not None:
            ref.next_step()
        ora.next_step()
        v = ora.vehicles()
        sample = list(zip(v["flow"], v["cnt"]))[:: max(1, len(v) // 7)]
        stats["leaders"] += len(sample)
        obs = observe_restatement(v, sample)
        if ref is not None:
            theirs = observe_reference(sample)
            assert theirs == obs, (s, [k for k in obs if obs[k] != theirs[k]])
            obs = theirs
        obs["rerouted"] = rerouted
        yield s, obs, dict(stats, vehicles=len(v))


# ---------------------------------------------------------------------------------------------------- recording
def _scenarios():
    sys.path.insert(0, HERE)
    import conftest
    return conftest


def _ref_trail(states, parts, group):
    t = Trail(parts, group)
    for st in states:
        t.add(st.step, st)
    t.close(states[-1].step)
    return t.pin()


def _save(name, doc):
    os.makedirs(PINS, exist_ok=True)
    with open(os.path.join(PINS, name + ".json"), "w") as f:
        json.dump(doc, f, sort_keys=True, separators=(",", ":"))
        f.write("\n")
    print(name, os.path.getsize(os.path.join(PINS, name + ".json")), "bytes")


def _save_blob(name, data: bytes):
    os.makedirs(PINS, exist_ok=True)
    with open(os.path.join(PINS, name + ".gz"), "wb") as f:
        f.write(gzip.compress(data, 9, mtime=0))


def _run(cfg, steps, every, threads=1):
    o = H.PortOracle(cfg)
    return H.RefDump.run(cfg, steps, threads, every, n_inter=o.n_inter, n_drivables=o.n_drivables)


def _runlc(cfg, steps, patched=True):
    o = H.PortOracle(cfg)
    return H.RefDump.runlc(cfg, steps, 1, n_inter=o.n_inter, n_drivables=o.n_drivables, patched=patched)


def record_examples(d, reference):
    """the reference's examples/ scenario (its roadnet and flow files are stored as they are)"""
    ex = os.path.join(reference, "examples")
    for f in ("roadnet.json", "flow.json"):
        data = open(os.path.join(ex, f), "rb").read()
        _save_blob("examples_" + f, data)
        open(os.path.join(d, f), "wb").write(data)
    cfg = json.load(open(os.path.join(ex, "config.json")))
    cfg["dir"] = d + "/"
    cfg["saveReplay"] = False
    p = os.path.join(d, "config.json")
    json.dump(cfg, open(p, "w"))
    run = _run(p, 300, 1)
    doc = _ref_trail(run, FULL + ("order",), 25)
    doc.update(config={k: v for k, v in cfg.items() if k != "dir"}, final_vehicles=run[-1].vehicle_count,
               final_lane_count_sum=int(run[-1].lane_count.sum()))
    _save("examples", doc)


def record_thread_count(d):
    cfg = _scenarios().cfg_3x3_dense.__wrapped__(d)
    _save("thread_count", {str(t): _ref_trail(_run(cfg, 200, 100, t), FULL + ("order",), 1) for t in (1, 4)})


def record_static_3x3(d):
    _save("static_3x3_dense", ref_static(_scenarios().cfg_3x3_dense.__wrapped__(d)))


def record_generator_tool(d, reference):
    import subprocess
    out = {}
    for rows, cols in ((1, 1), (2, 3), (6, 6)):
        subprocess.check_call([sys.executable, os.path.join(reference, "tools/generator/generate_grid_scenario.py"),
                               str(rows), str(cols), "--dir", d, "--roadnetFile", "r.json", "--flowFile", "f.json", "--tlPlan"])
        net = json.load(open(os.path.join(d, "r.json")))
        for i in net["intersections"]:
            for p in i["trafficLight"]["lightphases"]:
                p["availableRoadLinks"] = sorted(p["availableRoadLinks"])
        out["%dx%d" % (rows, cols)] = {"roadnet": value_digest(net), "flows": value_digest(json.load(open(os.path.join(d, "f.json"))))}
    _save("generator_tool", out)


def record_hetero(d):
    cfg = _scenarios().cfg_hetero_halfstep.__wrapped__(d)
    run = _run(cfg, 1500, 50)
    doc = _ref_trail(run, FULL + ("order",), 1)
    doc["final_finished"] = run[-1].finished
    _save("hetero_halfstep", doc)


def record_irregular(d):
    cfg = _scenarios().cfg_irregular.__wrapped__(d)
    run = _run(cfg, 600, 25)
    doc = _ref_trail(run, FULL + ("order",), 1)
    doc.update(static=ref_static(cfg), final_vehicles=run[-1].vehicle_count)
    _save("irregular", doc)


def record_replay(d):
    cfg = _scenarios().cfg_replay.__wrapped__(d)
    c = json.load(open(cfg))
    run = _run(cfg, 300, 30)
    lines = open(c["dir"] + c["replayLogFile"]).read().split("\n")
    doc = _ref_trail(run, ("vehicles", "phases"), 1)
    doc.update(lines=len(lines), roadnet_log=value_digest(json.load(open(c["dir"] + c["roadnetLogFile"]))))
    _save("replay", doc)
    _save_blob("replay_lines", "\n".join(replay_line_sample(lines[st.step - 1], st.step) for st in run).encode())


def replay_line_sample(line, step, k=48):
    """A replay step line shrunk to a seeded sample of k vehicle records (same positions on both sides), its light
    part and its number of vehicle records: "<n>|<record>,<record>,...;<lights>"."""
    va, lights = line.split(";")
    recs = va.split(",")
    pick = np.sort(np.random.default_rng(step).choice(len(recs), min(k, len(recs)), replace=False))
    return "%d|%s;%s" % (len(recs), ",".join(recs[i] for i in pick), lights)


def _lc_doc(run, group=25):
    doc = _ref_trail(run, LC, group)
    doc["shadows"] = int(sum((st.vehicles["partner_type"] == 2).sum() for st in run))
    return doc


def record_lane_change(d):
    from cityflow_b200 import scenario
    _scenarios()
    from test_cpu import _hetero_lane_change_config
    _save("lc_irregular", _lc_doc(_runlc(_hetero_lane_change_config(d), 900)))
    cfg = scenario.make_grid_scenario(d, 5, 5, dense=dict(frac=1.0, interval=2.0, seed=7), name="lc55", lane_change=True)
    _save("lc_5x5", _lc_doc(_runlc(cfg, 500)))


def record_lc_patch_neutral(d):
    import subprocess
    cfg = _scenarios().cfg_3x3_dense.__wrapped__(d)
    a, b = os.path.join(d, "a.bin"), os.path.join(d, "b.bin")
    subprocess.check_call([H.REFDUMP, "run", cfg, "300", "1", a, "1"])
    subprocess.check_call([H.REFDUMP_LC, "run", cfg, "300", "1", b, "1"])
    o = H.PortOracle(cfg)
    doc = {"unmodified": _ref_trail(H.parse_run(a, o.n_inter, o.n_drivables), FULL + ("order",), 25),
           "priority_ordered": _ref_trail(H.parse_run(b, o.n_inter, o.n_drivables), FULL + ("order",), 25)}
    doc["byte_identical"] = open(a, "rb").read() == open(b, "rb").read()
    _save("lc_patch_neutral", doc)


def lc_summary(states):
    started, seen, speed = 0, set(), []
    for st in states:
        sh = st.vehicles["priority"][st.vehicles["partner_type"] == 2]
        started += len(set(sh.tolist()) - seen)
        seen |= set(sh.tolist())
        speed.append(float(st.vehicles["speed"].mean()))
    return dict(finished=states[-1].finished, started=started, speed=float(np.mean(speed[200:])), vehicles=len(states[-1].vehicles))


def record_lc_statistics(d):
    from cityflow_b200 import scenario
    cfg = scenario.make_grid_scenario(d, 5, 5, dense=dict(frac=1.0, interval=2.0, seed=11), name="lcstat", lane_change=True)
    _save("lc_statistics", lc_summary(_runlc(cfg, 800, patched=False)))


def record_python_api(d):
    cfg = _scenarios().cfg_6x6_rl.__wrapped__(d)
    ref = H.load_reference_module().Engine(cfg, thread_num=1)
    ora = H.PortOracle(cfg)
    entries, _ = python_api_digests(python_api_run(ora, cfg, 520, ref))
    try:
        ref.set_vehicle_speed("flow_999999_0", 1.0)
        raised = False
    except RuntimeError:
        raised = True
    _save("python_api", {"entries": entries, "unknown_vehicle_raises": raised})


def random_network_config(directory, seed, interval, name, lane_change=False, n_flows=None, **shape):
    """tests/randnet.py network `seed` (its default size unless rows / cols are given) with flows from seed + 100"""
    sys.path.insert(0, HERE)
    import randnet
    from cityflow_b200 import scenario
    net = randnet.random_roadnet(seed, **shape)
    flows = randnet.random_flows(net, seed + 100, **({"n_flows": n_flows} if n_flows else {}))
    return scenario.write_scenario(directory, net, flows, seed=seed, interval=interval, lane_change=lane_change, name=name)


def record_random_networks(d):
    sys.path.insert(0, HERE)
    for seed, interval in ((1, 1.0), (2, 1.0), (3, 0.5), (4, 2.0), (5, 1.0), (6, 0.25)):
        cfg = random_network_config(d, seed, interval, "rand%d" % seed)
        run = _run(cfg, 700, 1)
        doc = _ref_trail(run, FULL + ("order",), 25)
        doc.update(static=ref_static(cfg), max_vehicles=max(s.vehicle_count for s in run), final_finished=run[-1].finished)
        _save("random_network_%d" % seed, doc)
    for seed in (17, 23):
        cfg = random_network_config(d, seed, [1.0, 0.5, 2.0, 1.0][seed % 4], "flc%d" % seed, True, 40 + seed % 50,
                                    rows=2 + seed % 3, cols=3 + seed % 2)
        _save("random_network_lc_%d" % seed, _lc_doc(_runlc(cfg, 400)))


def record_gpu_runs(d):
    cfg = _scenarios().cfg_6x6_dense.__wrapped__(d)
    _save("dense_6x6", _ref_trail(_run(cfg, 800, 20), GPU, 1))
    cfg = random_network_config(d, 4, 1.0, "gref", n_flows=70, rows=3, cols=4)
    _save("fuzzed_network_4", _ref_trail(_run(cfg, 500, 10, threads=2), GPU, 1))


def python_api_digests(run, group=10):
    """python_api_run's observations, one digest per `group` steps: ([{"steps": [first, last], "digest"}], final counters)"""
    out, h, stats = [], hashlib.sha256(), None
    for s, obs, stats in run:
        h.update(canonical(obs).encode())
        if s % group == 0:
            out.append({"steps": [s - group + 1, s], "digest": h.hexdigest()[:16]})
            h = hashlib.sha256()
    return out, stats


def bench_window_steps():
    """the steps test_30x30_through_the_bench_window_vs_compiled_reference compares the per-lane counts at"""
    return [s for s in range(10, 1231, 10) if s >= 1200 or s % 50 == 0]


def record_bench_window(d):
    from cityflow_b200 import scenario
    cfg = scenario.make_grid_scenario(d, 30, 30, name="g30w", dense=dict(frac=0.5, interval=10.0, seed=1, fleet_spread=0.02))
    ref = H.RefDump.counts(cfg, 1230, os.cpu_count() or 8, 10)
    lanes = {str(s): {"lane_count": lane_digest(ref["dumps"][s][0]), "lane_waiting": lane_digest(ref["dumps"][s][1])}
             for s in bench_window_steps()}
    cnt, _, ssum = ref["dumps"][1230]
    pick = np.sort(np.random.default_rng(1230).choice(ref["n_lanes"], 512, replace=False))
    counted = [s for s in range(1, 1231) if s >= 1200 or s % 5 == 0]
    _save("bench_window_30x30", {"vehicle_count": {str(s): int(ref["vehicle_count"][s - 1]) for s in counted}, "lanes": lanes,
                                 "n_lanes": ref["n_lanes"], "speed_sum_lanes": pick.tolist(), "speed_sum": [float(x) for x in ssum[pick]],
                                 "speed_sum_total": float(ssum.sum()), "vehicles_on_lanes": int(cnt.sum())})


def record_archives(d):
    """tests/archive_checks.py: the reference's JSON archive of the dense 3x3 run at step 120 (stored), its run after
    loading that file, and its runs after loading the files this engine writes (pinned by their bytes)."""
    import archive_checks
    from test_cpu import _emulated_engine
    os.environ["CFB_EMULATED_DEVICE_FOR_TESTS"] = "1"
    cf = _scenarios()
    cfg = cf.cfg_3x3_dense.__wrapped__(d)
    ours, theirs = os.path.join(d, "ours.json"), os.path.join(d, "ref.json")
    eng = _emulated_engine(cfg)
    eng.next_step(120)
    eng.dump(ours)
    H.RefDump.archive(cfg, 120, theirs)
    archive_checks.compare_archives(json.load(open(ours)), json.load(open(theirs)))
    kw = dict(n_inter=eng.n_inter, n_drivables=eng.n_drivables)
    from_ref, from_ours = H.RefDump.resume(cfg, theirs, 50, **kw), H.RefDump.resume(cfg, ours, 50, **kw)
    for a, b in zip(from_ref, from_ours):
        assert a.vehicle_count == b.vehicle_count and a.finished == b.finished and a.cum_travel_time == b.cum_travel_time
        assert a.vehicles.tobytes() == b.vehicles.tobytes(), a.step
    import lzma
    with open(os.path.join(PINS, "archive_3x3_dense_step120.json.xz"), "wb") as f:
        f.write(lzma.compress(open(theirs, "rb").read(), preset=9 | lzma.PRESET_EXTREME))
    doc = _ref_trail(from_ref, archive_checks.FOLLOW_PARTS, 1)
    doc["ours_resumed_identically"] = digest(open(ours, "rb").read())
    _save("archive_3x3_dense", doc)
    # rlTrafficLight: phases set right before the snapshot
    cfg = cf.cfg_6x6_rl.__wrapped__(d)
    eng = _emulated_engine(cfg)
    path, want = archive_checks.dump_with_rl_phases(eng, cfg, d)
    ref = H.RefDump.resume(cfg, path, 40, n_inter=eng.n_inter, n_drivables=eng.n_drivables)
    doc = _ref_trail(ref, archive_checks.FOLLOW_PARTS, 1)
    doc.update(ours=digest(open(path, "rb").read()), phases=[int(p) for p in ref[-1].phases if p >= 0])
    _save("archive_rl_6x6", doc)


def record_api_transcript(d):
    import api_parity_main
    cfg = _scenarios().cfg_6x6_rl.__wrapped__(d)
    _save("api_transcript", api_parity_main.record(H.load_reference_module(), cfg, 520))


# tests/test_gpu_multi.py: shard_rank_main.py arguments (rows cols steps every frac interval seed [fleet spread])
SHARD_RUNS = ([30, 60, 1230, 25, 0.5, 10, 1, 0.02], [8, 12, 400, 25, 1.0, 4, 1], [8, 12, 800, 25, 1.0, 4, 1],
              [30, 30, 600, 50, 0.5, 10, 1, 0.02])


def shard_run_key(args):
    return " ".join(str(a) for a in args)


def record_shard_runs(d):
    """the reference's collective observations behind tests/shard_rank_main.py: vehicle count after every step, per-lane
    vehicle and waiting counts every `every` steps (thread_num = host cores)"""
    from cityflow_b200 import scenario
    out = {}
    for a in SHARD_RUNS:
        rows, cols, steps, every, frac, interval, seed = a[:7]
        spread = a[7] if len(a) > 7 else 0.0
        cfg = scenario.make_grid_scenario(d, rows, cols, dense=dict(frac=frac, interval=interval, seed=seed, fleet_spread=spread), name="sh")
        ref = H.RefDump.counts(cfg, steps, os.cpu_count() or 8, every)
        out[shard_run_key(a)] = {"vehicle_count": {str(s): int(ref["vehicle_count"][s - 1]) for s in range(1, steps + 1)
                                                   if s % 5 == 0 or s == steps},
                                 "lanes": {str(s): {"lane_count": lane_digest(c), "lane_waiting": lane_digest(w)}
                                           for s, (c, w, _) in ref["dumps"].items()}}
    _save("shard_runs", out)


RECORDERS = {
    "examples": record_examples, "thread_count": record_thread_count, "static_3x3_dense": record_static_3x3,
    "generator_tool": record_generator_tool, "hetero_halfstep": record_hetero, "irregular": record_irregular,
    "replay": record_replay, "lane_change": record_lane_change, "lc_patch_neutral": record_lc_patch_neutral,
    "lc_statistics": record_lc_statistics, "python_api": record_python_api, "random_networks": record_random_networks,
    "gpu_runs": record_gpu_runs, "bench_window": record_bench_window, "archives": record_archives,
    "api_transcript": record_api_transcript, "shard_runs": record_shard_runs,
}


def main(names, reference):
    assert H.have_ref() and H.have_lc_ref(), "build the reference first: make -C oracle ref REF=<reference source tree>"
    if not H.have_port():
        H.build(ref=False)
    for name in names or list(RECORDERS):
        with tempfile.TemporaryDirectory() as d:
            fn = RECORDERS[name]
            fn(d, reference) if fn.__code__.co_argcount == 2 else fn(d)


if __name__ == "__main__":
    assert os.environ.get("REF"), "REF=<reference source tree> python tests/refpin.py [name ...]"
    main(sys.argv[1:], os.environ["REF"])
