"""GPU parity tests proper: the CUDA path, called through the C-ABI (ctypes), against the
checkers on identical seeded inputs -- the compiled unmodified reference (oracle/_ref/refdump),
through its pinned results (tests/refpin.py), and the CPU restatement (oracle/cityflow_oracle.cpp).

Bar (BASELINE.json north_star): per-lane vehicle counts bit-exact every step, per-vehicle speeds
within 1e-6.  What is asserted here is stronger: every running vehicle's (drivable, distance,
speed, leader, gap, blocker, enterLaneLinkTime) is bit-equal every step.
"""
import numpy as np
import pytest

import refpin
from oracle import harness as H

pytestmark = pytest.mark.gpu


def _gpu_state(eng, step):
    st = H.StepState()
    st.step = step
    st.vehicle_count = eng.vehicle_count()
    st.pool_size = st.finished = 0
    st.cum_travel_time = 0.0
    st.lane_count = eng.lane_vehicle_count()
    st.lane_waiting = eng.lane_waiting_count()
    st.lane_queue = None
    st.phases = None
    st.vehicles = eng.debug_vehicles()
    st.order = None
    return st


def _relax(ref):
    ref.pool_size = ref.finished = 0
    ref.cum_travel_time = 0.0
    return ref


def _run_against_port(cfg, steps, every=1, hook=None):
    from cityflow_b200.capi import CEngine
    eng = CEngine(cfg)
    ora = H.PortOracle(cfg)
    for s in range(1, steps + 1):
        if hook:
            hook(eng, ora, s)
        eng.next_step()
        ora.next_step()
        if s % every == 0 or s == steps:
            bad = H.compare_states(_relax(ora.snapshot()), _gpu_state(eng, s))
            assert not bad, "step %d: %s" % (s, "; ".join(bad[:6]))
    assert eng.gpu_launches() >= steps
    return eng, ora


def test_single_intersection_vs_port(cfg_1x1):
    _run_against_port(cfg_1x1, 300)


def test_3x3_dense_vs_port(cfg_3x3_dense):
    _run_against_port(cfg_3x3_dense, 600)


def test_6x6_default_vs_port(cfg_6x6):
    _run_against_port(cfg_6x6, 400, every=5)


def test_6x6_dense_vs_port(cfg_6x6_dense):
    eng, ora = _run_against_port(cfg_6x6_dense, 1200, every=10)
    assert ora.tie_count() == 0
    # finished vehicles and travel time bookkeeping (engine.cpp:299-303, :682-691): exact
    assert ora.lib.cfo_finished_count(ora.h) > 1000
    assert eng.average_travel_time() == ora.average_travel_time()


def test_rl_phases_vs_port(cfg_6x6_rl):
    # virtual intersections have no phases: the C-ABI rejects them, the oracle ignores them
    from cityflow_b200.capi import CEngine
    eng = CEngine(cfg_6x6_rl)
    ora = H.PortOracle(cfg_6x6_rl)
    ph0 = np.zeros(ora.n_inter, np.int32)
    ora.lib.cfo_phases(ora.h, ph0.ctypes.data)
    real = np.nonzero(ph0 >= 0)[0]
    for s in range(1, 401):
        if s % 10 == 1:
            for i in real:
                ph = int((s // 10 + i) % 8)
                eng.set_tl_phase(int(i), ph)
                ora.set_tl_phase(int(i), ph)
        eng.next_step()
        ora.next_step()
        if s % 5 == 0:
            bad = H.compare_states(_relax(ora.snapshot()), _gpu_state(eng, s))
            assert not bad, "step %d: %s" % (s, "; ".join(bad[:6]))


def test_6x6_dense_vs_compiled_reference(cfg_6x6_dense):
    from cityflow_b200.capi import CEngine
    eng = CEngine(cfg_6x6_dense)
    pin = refpin.load("dense_6x6")
    f = refpin.Follow(pin, parts=refpin.GPU, tag="6x6 dense")
    done = 0
    for _, step in pin["steps"]:        # every 20th step of 800
        eng.next_step(step - done)
        done = step
        f.add(done, _gpu_state(eng, done))
    f.finish()


def test_reset_determinism(cfg_3x3_dense):
    """The reference's own Basic.reset test (tests/cpp/basic_test.cpp:37-53)."""
    from cityflow_b200.capi import CEngine
    eng = CEngine(cfg_3x3_dense)
    eng.next_step(200)
    a = (eng.vehicle_count(), eng.lane_vehicle_count().copy(), eng.debug_vehicles().copy())
    eng.reset(True)
    eng.next_step(200)
    b = (eng.vehicle_count(), eng.lane_vehicle_count(), eng.debug_vehicles())
    assert a[0] == b[0]
    assert np.array_equal(a[1], b[1])
    assert np.array_equal(np.sort(a[2], order=["flow", "cnt"]), np.sort(b[2], order=["flow", "cnt"]))


def test_30x30_dense_lane_counts_vs_port(scenario_dir):
    """BASELINE.json configs[2] shape (30x30, dense demand): per-lane counts bit-exact and all
    speeds bit-equal against the CPU restatement while the network fills up."""
    from cityflow_b200 import scenario
    from cityflow_b200.capi import CEngine
    cfg = scenario.make_grid_scenario(scenario_dir, 30, 30, name="g30d", dense=dict(frac=0.5, interval=10.0, seed=1))
    eng = CEngine(cfg)
    ora = H.PortOracle(cfg)
    for s in (100, 250, 400):
        eng.next_step(s - ora.steps)
        ora.next_step(s - ora.steps)
        assert np.array_equal(eng.lane_vehicle_count(), ora.lane_vehicle_count()), "lane counts differ at step %d" % s
        assert np.array_equal(eng.lane_waiting_count(), ora.lane_waiting_count())
        bad = H.compare_states(_relax(ora.snapshot()), _gpu_state(eng, s))
        assert not bad, "step %d: %s" % (s, "; ".join(bad[:6]))
    assert ora.vehicle_count() > 50000


def _archive_record(eng, n):
    for _ in range(n):
        eng.next_step()
    return eng.get_lane_vehicle_count(), eng.get_average_travel_time(), eng.get_vehicle_speed()


def test_archive_snapshot_load_like_reference_tests(cfg_3x3_dense, tmp_path):
    """The reference's own result-pinning tests (tests/python/test_archive.py:16-23): run, snapshot,
    run 100 -> record, load, run 100 -> the record must be equal; also via dump / load_from_file and
    into a second engine built from the same config."""
    import cityflow
    eng = cityflow.Engine(cfg_3x3_dense, thread_num=1)
    for _ in range(150):
        eng.next_step()
    arc = eng.snapshot()
    rec1 = _archive_record(eng, 100)
    eng.load(arc)
    assert eng.get_current_time() == 150.0
    rec2 = _archive_record(eng, 100)
    assert rec1 == rec2
    # multiple loads of the same archive, and Archive(engine) constructor
    eng.load(arc)
    arc2 = cityflow.Archive(eng)
    assert _archive_record(eng, 100) == rec1
    eng.load(arc2)
    assert _archive_record(eng, 100) == rec1
    # file round trip into a fresh engine
    path = str(tmp_path / "save.bin")
    arc.dump(path)
    eng2 = cityflow.Engine(cfg_3x3_dense, thread_num=1)
    eng2.load_from_file(path)
    assert _archive_record(eng2, 100) == rec1


def test_vehicle_api_info_speed_route(cfg_3x3_dense):
    """SURVEY.md §8f-3 rows: get_vehicle_info / set_vehicle_speed / set_vehicle_route / get_leader."""
    import cityflow
    eng = cityflow.Engine(cfg_3x3_dense, thread_num=1)
    for _ in range(120):
        eng.next_step()
    speeds = eng.get_vehicle_speed()
    dist = eng.get_vehicle_distance()
    vid = next(k for k, v in speeds.items() if v > 3.0)
    info = eng.get_vehicle_info(vid)
    assert info["running"] == "1"
    assert float(info["speed"]) == pytest.approx(speeds[vid], abs=1e-6)
    assert float(info["distance"]) == pytest.approx(dist[vid], abs=1e-6)
    assert info["route"].endswith(" ") and "drivable" in info
    with pytest.raises(RuntimeError, match="not found"):
        eng.get_vehicle_info("flow_999999_0")
    with pytest.raises(RuntimeError, match="not found"):
        eng.set_vehicle_speed("nope", 1.0)
    # custom speed caps the next step's speed (Vehicle::getCarFollowSpeed, vehicle.cpp:214-221) for one step
    eng.set_vehicle_speed(vid, 0.5)
    eng.next_step()
    after = eng.get_vehicle_speed()
    if vid in after:
        assert after[vid] <= max(0.5, speeds[vid] - 4.5) + 1e-9
    leader = eng.get_leader(vid) if vid in after else ""
    assert isinstance(leader, str)
    # waiting vehicles are known but not running
    allv = eng.get_vehicles(include_waiting=True)
    run = set(eng.get_vehicles())
    assert run <= set(allv) and len(run) == eng.get_vehicle_count()
    lanes = eng.get_lane_vehicles()
    assert sum(len(v) for v in lanes.values()) == sum(eng.get_lane_vehicle_count().values())
    # re-routing: an unknown road or a vehicle on a laneLink is refused, a vehicle on a lane may keep its road
    assert eng.set_vehicle_route(vid, ["no_such_road"]) is False
    assert eng.set_vehicle_route("flow_999999_0", []) is False
    ok_any = False
    for cand, inf in ((k, eng.get_vehicle_info(k)) for k in list(after)[:200]):
        if "road" in inf:
            roads = inf["route"].split()
            if len(roads) >= 2:
                ok_any = eng.set_vehicle_route(cand, roads[1:2]) or ok_any
                break
    assert ok_any
    for _ in range(50):
        eng.next_step()
    assert eng.get_vehicle_count() > 0


def test_heterogeneous_vehicles_half_second_step_vs_port(cfg_hetero_halfstep):
    eng, ora = _run_against_port(cfg_hetero_halfstep, 1500, every=10)
    assert ora.vehicle_count() > 300


def test_push_vehicle_rng_interleaving_vs_port(cfg_3x3_dense):
    """push_vehicle draws its priority from the engine RNG at call time, i.e. between the flow
    draws of two steps (engine.cpp:693-717): the whole future then depends on the interleaving."""
    import json
    import os
    import cityflow
    cfgj = json.load(open(cfg_3x3_dense))
    flows = json.load(open(os.path.join(cfgj["dir"], cfgj["flowFile"])))
    route = flows[0]["route"][:3]
    eng = cityflow.Engine(cfg_3x3_dense, thread_num=1)
    ora = H.PortOracle(cfg_3x3_dense)
    for s in range(1, 301):
        if s % 7 == 0:
            info = {"speed": 0.0, "length": 6.0, "maxSpeed": 12.0} if s % 14 == 0 else {}
            eng.push_vehicle(info, route)
            ora.push_vehicle(info, route)
        eng.next_step()
        ora.next_step()
        if s % 25 == 0:
            assert eng.get_vehicle_count() == ora.vehicle_count()
            assert sum(eng.get_lane_vehicle_count().values()) == int(ora.lane_vehicle_count().sum())
            ov = ora.vehicles()
            sp = eng.get_vehicle_speed()
            names = ["flow_%d_%d" % (f, c) if f >= 0 else "manually_pushed_%d" % c for f, c in zip(ov["flow"], ov["cnt"])]
            assert set(names) == set(sp.keys())
            assert all(sp[n] == v for n, v in zip(names, ov["speed"]))
            assert eng.get_average_travel_time() == ora.average_travel_time()
    assert any(k.startswith("manually_pushed_") for k in sp)


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_loopback_equals_unsharded(cfg_6x6_dense, world):
    """SURVEY.md §8e exactness requirement: the network cut into `world` column strips (ranks on one
    GPU, seam exchanges by device copies) evolves bit-identically to the unsharded engine."""
    from cityflow_b200.capi import CEngine, CShardGroup
    ref = CEngine(cfg_6x6_dense)
    grp = CShardGroup(cfg_6x6_dense, world)
    for s in range(1, 801):
        ref.next_step()
        grp.next_step()
        if s % 20 == 0 or s < 40:
            assert grp.vehicle_count() == ref.vehicle_count(), "step %d" % s
            assert np.array_equal(grp.lane_counts(ref.n_lanes), ref.lane_vehicle_count()), "lane counts differ at step %d" % s
        if s % 100 == 0:
            assert np.array_equal(grp.lane_counts(ref.n_lanes, True), ref.lane_waiting_count())
            a = np.sort(ref.debug_vehicles(), order=["flow", "cnt"])
            b = np.sort(grp.debug_vehicles(), order=["flow", "cnt"])
            assert len(a) == len(b)
            for f in ("flow", "cnt", "drivable", "blocker_flow", "blocker_cnt", "enter_ll_time"):
                assert np.array_equal(a[f], b[f]), (s, f)
            for f in ("dis", "speed"):
                assert np.array_equal(a[f], b[f]), (s, f)
    assert ref.vehicle_count() > 3000


def test_priority_collisions_after_reseed_vs_port(cfg_3x3_dense):
    """Re-seeding the engine RNG mid-run makes it re-issue the priorities it drew at the start:
    draws collide with vehicles that are still alive (redraw, vehicle.cpp:45) and re-use the
    priorities of vehicles that already left (legal).  Exercises Engine::checkPriority
    (engine.cpp:601) against the host's lazily drained bookkeeping."""
    import cityflow
    eng = cityflow.Engine(cfg_3x3_dense, thread_num=1)
    ora = H.PortOracle(cfg_3x3_dense)
    for s in range(1, 701):
        if s in (250, 400, 401, 550):
            eng.set_random_seed(0)
            ora.set_random_seed(0)
        eng.next_step()
        ora.next_step()
        if s % 50 == 0 or s in (251, 252, 402):
            assert eng.get_vehicle_count() == ora.vehicle_count(), s
            ov = ora.vehicles()
            sp = eng.get_vehicle_speed()
            names = ["flow_%d_%d" % (f, c) for f, c in zip(ov["flow"], ov["cnt"])]
            assert set(names) == set(sp.keys()), s
            assert all(sp[n] == v for n, v in zip(names, ov["speed"])), s
    assert eng.get_average_travel_time() == ora.average_travel_time()


def test_irregular_roadnet_vs_port(cfg_irregular):
    _run_against_port(cfg_irregular, 600, every=10)


def test_device_resident_lane_observations(cfg_6x6_dense):
    """SURVEY.md §8f-3 zero-copy observations: the torch CUDA tensors alias the engine's buffers and
    carry exactly what the host getters report, refreshed without a host synchronisation."""
    import torch
    import cityflow
    import cityflow_b200
    eng = cityflow.Engine(cfg_6x6_dense, thread_num=1)
    side = torch.cuda.Stream()
    for rounds in range(3):
        for _ in range(100):
            eng.next_step()
        with torch.cuda.stream(side if rounds == 1 else torch.cuda.current_stream()):
            ids, cnt, wait, ssum = cityflow_b200.lane_observation_tensors(eng)
            total = cnt.sum()                               # consumer work on the ordered stream
            cnt_h, wait_h, ssum_h = cnt.cpu(), wait.cpu(), ssum.cpu()
        assert cnt.is_cuda and cnt.dtype == torch.int32 and ssum.dtype == torch.float64
        counts = eng.get_lane_vehicle_count()
        waiting = eng.get_lane_waiting_vehicle_count()
        assert ids == eng.lane_ids() and set(ids) == set(counts)
        assert cnt_h.tolist() == [counts[i] for i in ids]
        assert wait_h.tolist() == [waiting[i] for i in ids]
        assert int(total) == sum(counts.values())
        speeds = eng.get_vehicle_speed()
        per_lane = {i: 0.0 for i in ids}
        for lane, vs in eng.get_lane_vehicles().items():
            per_lane[lane] = sum(speeds[v] for v in vs)
        np.testing.assert_allclose(ssum_h.numpy(), np.array([per_lane[i] for i in ids]), rtol=0, atol=1e-9)
    assert sum(counts.values()) > 500
    # same storage every call (zero-copy): the next refresh shows through the old tensor
    old_ptr = cnt.data_ptr()
    eng.next_steps(50)
    ids2, cnt2, _, _ = cityflow_b200.lane_observation_tensors(eng)
    assert cnt2.data_ptr() == old_ptr
    assert cnt.tolist() == [eng.get_lane_vehicle_count()[i] for i in ids]
    # the persistent form: tensors made once, refresh() only re-computes their content
    obs = cityflow_b200.LaneObservations(eng)
    eng.next_steps(25)
    before = obs.vehicle_count.clone()
    assert obs.refresh() is obs and obs.vehicle_count.data_ptr() == old_ptr
    now = eng.get_lane_vehicle_count()
    assert obs.vehicle_count.tolist() == [now[i] for i in obs.lane_ids]
    assert not torch.equal(before, obs.vehicle_count)


def test_rl_actions_and_observations_on_device_vs_port(cfg_6x6_rl):
    """The RL loop with nothing crossing to the host: actions come from a torch tensor
    (cfb_set_tl_phases_device), observations are torch tensors; the oracle gets the same actions
    through its host API and must see the same lane counts every step."""
    import torch
    import cityflow
    import cityflow_b200
    eng = cityflow.Engine(cfg_6x6_rl, thread_num=1)
    ora = H.PortOracle(cfg_6x6_rl)
    ph0 = np.zeros(ora.n_inter, np.int32)
    ora.lib.cfo_phases(ora.h, ph0.ctypes.data)
    real = np.nonzero(ph0 >= 0)[0]
    assert eng.num_intersections() == ora.n_inter
    idx = torch.arange(ora.n_inter, device="cuda", dtype=torch.int32)
    for s in range(1, 301):
        if s % 10 == 1:
            act = ((s // 10 + idx) % 8).to(torch.int32)       # computed on the GPU, never copied down
            cityflow_b200.set_tl_phases_tensor(eng, act)
            del act
            for i in real:
                ora.set_tl_phase(int(i), int((s // 10 + i) % 8))
        eng.next_step()
        ora.next_step()
        if s % 5 == 0:
            ids, cnt, wait, _ = cityflow_b200.lane_observation_tensors(eng)
            snap = ora.snapshot()
            assert cnt.cpu().numpy().tolist() == list(snap.lane_count)
            assert wait.cpu().numpy().tolist() == list(snap.lane_waiting)
    assert int(cnt.sum()) > 300
    # host-side set_tl_phase after a device-side one starts from the device's phases
    some = eng.intersection_ids()[int(real[0])]
    eng.set_tl_phase(some, 3)
    ora.set_tl_phase(int(real[0]), 3)
    for _ in range(40):
        eng.next_step()
        ora.next_step()
    counts = eng.get_lane_vehicle_count()
    assert [counts[i] for i in ids] == list(ora.snapshot().lane_count)
    # an out-of-range action is reported (the reference would throw from phases.at())
    bad = torch.full((ora.n_inter,), 99, device="cuda", dtype=torch.int32)
    cityflow_b200.set_tl_phases_tensor(eng, bad)
    eng.next_step()
    with pytest.raises(RuntimeError, match="out of range"):
        for _ in range(300):          # surfaced by the next bookkeeping drain at the latest
            eng.next_step()
        eng.get_average_travel_time()


def test_replay_files_written_by_the_engine(cfg_replay):
    """SURVEY.md §8f-4: with saveReplay the engine writes the reference's two log files.  The step
    lines must be exactly what the stand-alone formatter makes of the ORACLE's states (so: device
    positions, priority order and light states all agree); tests/test_cpu.py pins that formatter
    against the files the compiled reference writes."""
    import json
    import os
    import cityflow
    from cityflow_b200.capi import CReplay, REPLAY_DTYPE
    c = json.load(open(cfg_replay))
    log, netlog, log2 = c["dir"] + c["replayLogFile"], c["dir"] + c["roadnetLogFile"], c["dir"] + "replay_second.txt"
    for f in (log, netlog, log2):
        if os.path.exists(f):
            os.remove(f)
    flows = json.load(open(c["dir"] + c["flowFile"]))
    eng = cityflow.Engine(cfg_replay, thread_num=1)
    ora = H.PortOracle(cfg_replay)
    rp = CReplay(c["dir"] + c["roadnetFile"])
    assert open(netlog).read() == rp.roadnet_json()
    expect = []
    for s in range(1, 201):
        if s == 151:
            eng.set_save_replay(False)          # engine.cpp:736-742: steps 151..160 leave no line
        if s == 161:
            eng.set_save_replay(True)
            eng.set_replay_file("replay_second.txt")   # engine.cpp:727-734: relative to "dir"
        eng.next_step()
        ora.next_step()
        st = ora.snapshot()
        v = np.zeros(len(st.vehicles), REPLAY_DTYPE)
        v["drivable"], v["distance"] = st.vehicles["drivable"], st.vehicles["dis"]
        v["flow"], v["index"] = st.vehicles["flow"], st.vehicles["cnt"]
        v["length"] = [flows[f]["vehicle"]["length"] for f in st.vehicles["flow"]]
        v["width"] = [flows[f]["vehicle"]["width"] for f in st.vehicles["flow"]]
        expect.append(rp.format_step(v, np.where(st.phases < 0, 0, st.phases)))
    del eng                                      # closes the log like ~Engine (engine.cpp:763)
    first = open(log).read().split("\n")
    second = open(log2).read().split("\n")
    assert first[-1] == "" and second[-1] == ""
    assert first[:-1] == expect[:150]
    assert second[:-1] == expect[160:]
    assert len(expect[-1].split(",")) > 100


def _lc_gpu_states(eng, steps):
    """Per-step LC_DTYPE records of the GPU engine (every running vehicle including shadows) as StepState objects."""
    import ctypes
    lib = eng.lib
    lib.cfb_debug_lc_vehicles.restype = ctypes.c_int64
    lib.cfb_debug_lc_vehicles.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]
    lib.cfb_finished_vehicle_count.restype = ctypes.c_int64
    lib.cfb_finished_vehicle_count.argtypes = [ctypes.c_void_p]
    out = []
    for _ in range(steps):
        eng.next_step()
        n = int(lib.cfb_debug_lc_vehicles(eng.h, None, 0))
        got = np.zeros(n, H.LC_DTYPE)
        if n:
            lib.cfb_debug_lc_vehicles(eng.h, got.ctypes.data, n)
        st = H.StepState()
        st.vehicles = got
        st.finished = int(lib.cfb_finished_vehicle_count(eng.h))
        out.append(st)
    return out


def test_lane_change_statistics_vs_unmodified_reference(tmp_path):
    """laneChange=true against the UNMODIFIED reference.  Its lane-change schedule follows heap addresses (the order of
    a std::set<Vehicle*>), so only aggregates can agree: vehicles that finished, lane changes started, mean speed, running
    vehicles -- same tolerances as the restatement's own comparison (tests/test_cpu.py)."""
    from cityflow_b200 import scenario
    from cityflow_b200.capi import CEngine
    cfg = scenario.make_grid_scenario(str(tmp_path), 5, 5, dense=dict(frac=1.0, interval=2.0, seed=11), name="lcstat", lane_change=True)
    eng = CEngine(cfg)
    a, b = refpin.load("lc_statistics"), refpin.lc_summary(_lc_gpu_states(eng, 800))
    assert a["started"] > 200 and b["started"] > 200, (a, b)
    for k, tol in (("finished", 0.03), ("started", 0.15), ("speed", 0.03), ("vehicles", 0.03)):
        assert abs(a[k] - b[k]) <= tol * a[k], (k, a, b)


def test_lane_change_vs_restatement(tmp_path):
    """laneChange=true on the GPU against the restatement (pinned to oracle/_ref/refdump_lcorder, the reference with its
    worker sets ordered by priority): every running vehicle including shadows, every field, every step."""
    import ctypes
    from cityflow_b200 import scenario
    from cityflow_b200.capi import CEngine
    cfg = scenario.make_grid_scenario(str(tmp_path), 4, 4, dense=dict(frac=1.0, interval=3.0, seed=2), name="lc", lane_change=True)
    eng, ora = CEngine(cfg), H.PortOracle(cfg)
    lib = eng.lib
    lib.cfb_debug_lc_vehicles.restype = ctypes.c_int64
    lib.cfb_debug_lc_vehicles.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]
    shadows = 0
    for s in range(1, 401):
        eng.next_step()
        ora.next_step()
        want = ora.lc_snapshot()
        n = int(lib.cfb_debug_lc_vehicles(eng.h, None, 0))
        got = np.zeros(n, H.LC_DTYPE)
        if n:
            lib.cfb_debug_lc_vehicles(eng.h, got.ctypes.data, n)
        assert eng.vehicle_count() == want.vehicle_count, "step %d" % s
        assert np.array_equal(eng.lane_vehicle_count(), want.lane_count), "lane counts, step %d" % s
        assert len(got) == len(want.vehicles), "step %d" % s
        for f in H.LC_DTYPE.names:
            assert np.array_equal(got[f], want.vehicles[f]), "step %d field %s" % (s, f)
        shadows += int((want.vehicles["partner_type"] == 2).sum())
    assert shadows > 300


# ------------------------------------------------------------------------------------------
# Irregular networks (tests/randnet.py): missing streets, 1-3 lanes, bent roads, sparse laneLink sets -- including first
# lanes that cannot continue the route two roads ahead, where Vehicle::getNextSpeed's `if (laneChange)` block
# (vehicle.cpp:323-329, it tests the LaneChange OBJECT and so runs with laneChange=false too) parks the vehicle at the end
# of the lane.  Full state every step against the restatement (which is pinned to the compiled reference on the same
# generator, tests/test_cpu.py::test_random_network_loader_and_oracle_vs_reference).
@pytest.mark.parametrize("seed", [1, 2, 3, 5, 8, 11])
def test_fuzzed_irregular_networks_vs_port(seed, tmp_path):
    import randnet
    from cityflow_b200 import scenario
    net = randnet.random_roadnet(seed, rows=2 + seed % 3, cols=3 + seed % 2)
    flows = randnet.random_flows(net, seed + 100, n_flows=40 + seed % 50)
    cfg = scenario.write_scenario(str(tmp_path), net, flows, seed=seed, interval=[1.0, 0.5, 2.0, 1.0][seed % 4], name="g%d" % seed)
    _run_against_port(cfg, 500)


def test_fuzzed_network_vs_compiled_reference(tmp_path):
    """The same kind of network straight against the UNMODIFIED reference (oracle/_ref/refdump): the restatement shares the
    product's loader, the compiled reference does not -- a loader / routing bug cannot hide behind it here."""
    from cityflow_b200.capi import CEngine
    cfg = refpin.random_network_config(str(tmp_path), 4, 1.0, "gref", n_flows=70, rows=3, cols=4)
    eng = CEngine(cfg)
    pin = refpin.load("fuzzed_network_4")     # reference with thread_num=2, every 10th step of 500
    f = refpin.Follow(pin, parts=refpin.GPU, tag="fuzzed network 4")
    done = 0
    for _, step in pin["steps"]:
        eng.next_step(step - done)
        done = step
        f.add(done, _gpu_state(eng, done))
    f.finish()
    assert eng.tie_count() == 0


def test_vehicle_setters_step_by_step_vs_port(tmp_path):
    """set_vehicle_speed / set_vehicle_route (engine.cpp:827-866) applied identically to the GPU engine and to the
    restatement (itself pinned to the reference's Python module): every speed of every vehicle after every step."""
    import json
    import os
    import cityflow
    from cityflow_b200 import scenario
    cfg = scenario.make_grid_scenario(str(tmp_path), 4, 4, dense=dict(frac=1.0, interval=3.0, seed=2), name="api")
    flows = json.load(open(os.path.join(str(tmp_path), "flow_api.json")))
    eng, ora = cityflow.Engine(cfg, thread_num=1), H.PortOracle(cfg)

    def vid(f, k):
        return "manually_pushed_%d" % k if f == -2 else "flow_%d_%d" % (f, k)

    for s in range(1, 401):
        v = ora.vehicles()
        if s % 20 == 3:
            for j in range(0, len(v), max(1, len(v) // 6)):
                f, k, sp = int(v["flow"][j]), int(v["cnt"][j]), float(v["speed"][j]) * 0.5
                eng.set_vehicle_speed(vid(f, k), sp)
                assert ora.set_vehicle_speed(f, k, sp)
        if s % 30 == 7:
            for j in range(1, len(v), max(1, len(v) // 8)):
                f, k = int(v["flow"][j]), int(v["cnt"][j])
                target = flows[(s + j) % len(flows)]["route"][-1:]
                assert eng.set_vehicle_route(vid(f, k), target) == ora.set_vehicle_route(f, k, target), (s, vid(f, k))
        eng.next_step()
        ora.next_step()
        v = ora.vehicles()
        mine = eng.get_vehicle_speed()
        theirs = {vid(f, k): sp for f, k, sp in zip(v["flow"], v["cnt"], v["speed"])}
        assert mine == theirs, "step %d: %s" % (s, [(k, mine.get(k), theirs[k]) for k in theirs if mine.get(k) != theirs[k]][:3])


def test_30x30_through_the_bench_window_vs_compiled_reference(scenario_dir):
    """The bench operating point itself: BASELINE.json configs[2] (30x30, ~1.3e5 vehicles, gridlock) against the UNMODIFIED
    reference -- vehicle count after every step, per-lane counts, per-lane waiting counts (speed < 0.1) and per-lane speed
    sums (within 1e-6 per vehicle) every 50 steps and at steps 1200, 1210, 1220, 1230 (the vehicle count at every step of
    the window 1200..1230)."""
    from cityflow_b200 import scenario
    from cityflow_b200.capi import CEngine
    cfg = scenario.make_grid_scenario(scenario_dir, 30, 30, name="g30w", dense=dict(frac=0.5, interval=10.0, seed=1, fleet_spread=0.02))
    ref = refpin.load("bench_window_30x30")   # the reference with thread_num = host cores
    assert ref["lanes"].keys() == {str(s) for s in refpin.bench_window_steps()}
    eng = CEngine(cfg)
    for s in range(1, 1231):
        eng.next_step()
        if s >= 1200 or s % 5 == 0:
            assert eng.vehicle_count() == ref["vehicle_count"][str(s)], s
        if str(s) not in ref["lanes"]:
            continue
        mc, mw = eng.lane_vehicle_count(), eng.lane_waiting_count()
        assert refpin.lane_digest(mc) == ref["lanes"][str(s)]["lane_count"], "step %d: lane counts differ" % s
        assert refpin.lane_digest(mw) == ref["lanes"][str(s)]["lane_waiting"], "step %d: lane waiting counts differ" % s
    # per-vehicle speeds at the end, through the per-lane speed sums (bar: 1e-6 per vehicle; the sums differ by summation order
    # only): on a seeded sample of 512 lanes, and in total
    v = eng.debug_vehicles()
    on = v[v["drivable"] < eng.n_lanes]
    mine = np.bincount(on["drivable"], weights=on["speed"], minlength=eng.n_lanes)
    pick, rs = np.array(ref["speed_sum_lanes"]), np.array(ref["speed_sum"])
    assert eng.n_lanes == ref["n_lanes"] and int(mc.sum()) == ref["vehicles_on_lanes"]
    assert np.all(np.abs(mine[pick] - rs) <= 1e-6 * np.maximum(mc[pick], 1)), "per-lane speed sums differ"
    assert abs(mine.sum() - ref["speed_sum_total"]) <= 1e-6 * int(mc.sum()), "speed sum over all lanes differs"
    assert eng.vehicle_count() > 120000
    assert eng.tie_count() == 0   # (the bench fleet: no entrant tie, so the reference's result is defined -- bench.py FLEET_SPREAD)


def test_6x6_3600_steps_vs_port(cfg_6x6):
    """BASELINE.json configs[1] length: the generator's default 6x6 scenario for the full 3600 steps, full state every 100."""
    _run_against_port(cfg_6x6, 3600, every=100)
