"""Checks of the reference-schema JSON archive (Archive::dump archive.cpp:153-343, the file loader :345-550) shared by the
CPU test (the real host engine over the emulated device, tests/test_cpu.py) and the GPU test (tests/test_gpu_zarchive.py).
TEST INFRASTRUCTURE: the checker is the UNMODIFIED reference (oracle/_ref/refdump, modes `archive` and `resume`), through
what it computed on these scenarios (tests/refpin.py, tests/golden/reference/): its own archive file, its runs after
loading that file and after loading the files this engine writes.

What "equal" means here.  The reference's own file round trip is lossy: its JSON parser (rapidjson without
kParseFullPrecisionFlag) returns some 17-digit numbers one ulp off, so an engine that loads a file does NOT continue the
uninterrupted trajectory -- in the reference itself.  The parity target is therefore the reference LOADING THE SAME FILE:
this engine's loader parses numbers the way rapidjson does (csrc/json_min.h), and must then move every vehicle exactly
as the reference does after its loadFromFile()."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle import harness as H   # noqa: E402
import refpin   # noqa: E402

STATE_FIELDS = ("flow", "cnt", "priority", "drivable", "dis", "speed", "leader_flow", "leader_cnt", "blocker_flow", "blocker_cnt", "gap")
FOLLOW_PARTS = ("vehicle_count", "lane_count", "lane_waiting", "state")   # refpin parts of what follow() compares


def compare_archives(ours: dict, ref: dict):
    """Every member of every vehicle, drivable, flow and light.  (`refdump archive` first gives the two members the
    reference leaves uninitialised -- `gap` without a leader, `enterLaneLinkTime` before the first change of drivable --
    the values this engine writes, see oracle/refdump.cpp; the lanes' speed history is written empty here: it is read
    only by RouterType::DURATION routing, which nothing in the engine selects.)"""
    assert sorted(ours) == sorted(ref)
    for k in ("step", "activeVehicleCount", "rnd", "finishedVehicleCnt", "cumulativeTravelTime", "flows", "trafficLights"):
        assert ours[k] == ref[k], k
    assert [v["id"] for v in ours["vehicles"]] == [v["id"] for v in ref["vehicles"]]      # priority order
    checked = 0
    for a, b in zip(ours["vehicles"], ref["vehicles"]):
        assert sorted(a) == sorted(b), (a["id"], sorted(a), sorted(b))
        for k in a:
            assert a[k] == b[k], (a["id"], k, a[k], b[k])
            checked += 1
    assert sorted(ours["drivables"]) == sorted(ref["drivables"])
    for d, x in ours["drivables"].items():
        y = ref["drivables"][d]
        assert sorted(x) == sorted(y), d
        assert x["vehicles"] == y["vehicles"], d
        assert x.get("waitingBuffer") == y.get("waitingBuffer"), d
    return checked


def follow(eng, pin, tag):
    """`eng` steps along the reference's pinned states: vehicle count, per-lane counts and waiting counts, and every
    running vehicle in every field of STATE_FIELDS, every step."""
    f = refpin.Follow(pin, tag=tag)
    g = None
    for a, b in pin["steps"]:
        for s in range(a, b + 1):
            eng.next_step()
            st = H.StepState()
            st.vehicle_count = eng.vehicle_count()
            st.lane_count, st.lane_waiting = eng.lane_vehicle_count(), eng.lane_waiting_count()
            st.vehicles = g = eng.debug_vehicles()
            f.add(s, st)
    f.finish()
    return g


def check_json_interchange(make_engine, cfg: str, tmp: str):
    """Both directions at step 120 of the dense 3x3 scenario, followed for 50 steps:
    (1) this engine's dump equals the reference's own dump field by field, and it is the file the reference was seen to
        load and then move exactly as from its own file; (2) this engine loads the reference's file -- over an unrelated
        state -- and then moves exactly as the reference does from that file; (3) the file written here loads back here to
        the same trajectory as (2), travel-time statistics included."""
    import lzma
    pin = refpin.load("archive_3x3_dense")
    ours_path, ref_path = os.path.join(tmp, "ours.json"), os.path.join(tmp, "ref.json")
    with open(os.path.join(refpin.PINS, "archive_3x3_dense_step120.json.xz"), "rb") as f, open(ref_path, "wb") as g:
        g.write(lzma.decompress(f.read()))
    eng = make_engine(cfg)
    eng.next_step(120)
    eng.dump(ours_path)
    checked = compare_archives(json.load(open(ours_path)), json.load(open(ref_path)))
    assert checked > 20000
    assert refpin.digest(open(ours_path, "rb").read()) == pin["ours_resumed_identically"], \
        "the archive is not the file the reference was seen to resume like its own (re-record with tests/refpin.py archives)"
    # (2) the reference's file into an engine that is somewhere else entirely
    other = make_engine(cfg)
    other.next_step(17)
    other.load_from_file(ref_path)
    g = follow(other, pin, "reference file")
    assert len(g) > 300
    # (3) our own file back into the first engine (it has moved on in the meantime)
    eng.next_step(5)
    eng.load_from_file(ours_path)
    follow(eng, pin, "own file")
    assert eng.average_travel_time() == other.average_travel_time()


def dump_with_rl_phases(eng, cfg: str, tmp: str):
    """90 steps, then a phase for every signalised intersection and at once snapshot().dump("rl.json")."""
    roadnet = json.load(open(json.load(open(cfg))["dir"] + json.load(open(cfg))["roadnetFile"]))
    real = [k for k, i in enumerate(roadnet["intersections"]) if not i["virtual"]]
    eng.next_step(90)
    want = {k: (3 * n + 1) % 8 for n, k in enumerate(real)}
    for k, ph in want.items():
        eng.set_tl_phase(k, ph)
    path = os.path.join(tmp, "rl.json")
    eng.dump(path)
    doc = json.load(open(path))
    assert doc["step"] == 90 and doc["activeVehicleCount"] == eng.vehicle_count()
    for k, ph in want.items():
        assert doc["trafficLights"][roadnet["intersections"][k]["id"]]["curPhaseIndex"] == ph
    return path, [want[k] for k in real]


def check_json_with_rl_phases(make_engine, cfg: str, tmp: str):
    """rlTrafficLight mode, phases set right before the snapshot (not yet sent to the device when it is taken): the file
    carries them, the reference resuming from it showed them and moved the vehicles as this engine does after loading the
    same file."""
    pin = refpin.load("archive_rl_6x6")
    path, want = dump_with_rl_phases(make_engine(cfg), cfg, tmp)
    assert refpin.digest(open(path, "rb").read()) == pin["ours"], \
        "the archive is not the file the reference was seen to resume (re-record with tests/refpin.py archives)"
    assert pin["phases"] == want
    other = make_engine(cfg)
    other.load_from_file(path)
    follow(other, pin, "rl file")


def check_reference_disk_io_tests(make_engine, cfg: str, tmp: str, record):
    """The reference's own tests/python/test_archive.py:95-119 (test_save_to_file, test_multi_save_to_file), file name
    included: dump("save.json") after 100 steps, 100 more -> record, load_from_file("save.json"), 100 steps -> the
    same record (lane vehicle counts + average travel time), twice over.  `cfg` must be a scenario whose routes visit
    no road twice: on other routes the reference's reloaded router deviates (see Routing::planFrom) and its own test
    would fail."""
    path = os.path.join(tmp, "save.json")
    eng = make_engine(cfg)
    for _ in range(2):
        eng.next_step(100)
        eng.dump(path)
        assert open(path).read(1) == "{"
        eng.next_step(100)
        want = record(eng)
        for _ in range(2):
            eng.load_from_file(path)
            eng.next_step(100)
            assert record(eng) == want


def lc_vehicles(eng):
    """cfb_debug_lc_vehicles: every running vehicle incl. shadows with its lane-change state."""
    import ctypes
    lib = eng.lib
    lib.cfb_debug_lc_vehicles.restype = ctypes.c_int64
    lib.cfb_debug_lc_vehicles.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]
    n = int(lib.cfb_debug_lc_vehicles(eng.h, None, 0))
    got = np.zeros(n, H.LC_DTYPE)
    if n:
        lib.cfb_debug_lc_vehicles(eng.h, got.ctypes.data, n)
    return got


def check_lane_change_snapshot(make_engine, cfg: str, tmp: str):
    """laneChange = true: the binary archive carries the per-vehicle lane-change state (partners, offsets, signals,
    waiting times).  Taken while shadows are on the road, loaded into the same and into a fresh engine: the
    uninterrupted run, every field of every vehicle and shadow, 60 steps.  The JSON form is refused with laneChange."""
    eng = make_engine(cfg)
    eng.next_step(100)
    for _ in range(200):
        if (lc_vehicles(eng)["partner_type"] == 2).sum() >= 2:
            break
        eng.next_step()
    assert (lc_vehicles(eng)["partner_type"] == 2).sum() >= 2
    path = os.path.join(tmp, "lc.bin")
    eng.dump(path)
    want = []
    for _ in range(60):
        eng.next_step()
        want.append((eng.vehicle_count(), lc_vehicles(eng).tobytes()))
    fresh = make_engine(cfg)
    for e in (eng, fresh):
        e.load_from_file(path)
        for k in range(60):
            e.next_step()
            assert (e.vehicle_count(), lc_vehicles(e).tobytes()) == want[k], k
    try:
        eng.dump(os.path.join(tmp, "lc.json"))
        raise AssertionError("the JSON form must be refused with laneChange on")
    except RuntimeError as ex:
        assert "laneChange" in str(ex)


def check_damaged_json_is_refused(make_engine, cfg: str, tmp: str, rounds: int = 150, seed: int = 1):
    """load_from_file on damaged input: a valid archive with random structural damage (members removed or retyped, list
    entries removed / duplicated / replaced, truncation).  Every file is either refused with an error or accepted and
    steppable, never a crash, and the engine loads the intact file afterwards."""
    import copy
    import random
    rng = random.Random(seed)
    eng = make_engine(cfg)
    eng.next_step(80)
    good, bad = os.path.join(tmp, "good.json"), os.path.join(tmp, "bad.json")
    eng.dump(good)
    doc = json.load(open(good))

    def mutate(x, depth=0):
        if isinstance(x, dict) and x:
            k = rng.choice(list(x))
            r = rng.random()
            if r < 0.25 or depth > 3:
                del x[k]
            elif r < 0.5:
                x[k] = rng.choice([None, -1, 1e308, "zzz", [], {}, True, 2 ** 40, -2 ** 40, "road_0_0_0", 1.5])
            elif not mutate(x[k], depth + 1):
                x[k] = rng.choice([None, -5, "x", [], {}])
            return True
        if isinstance(x, list) and x:
            i = rng.randrange(len(x))
            r = rng.random()
            if r < 0.2:
                del x[i]
            elif r < 0.4:
                x.append(copy.deepcopy(x[i]))
            elif r < 0.6:
                x[i] = rng.choice([None, 7, "flow_0_0", "nope", {}, []])
            elif not mutate(x[i], depth + 1):
                x[i] = rng.choice([None, -5, "x"])
            return True
        return False

    refused = 0
    for _ in range(rounds):
        m = copy.deepcopy(doc)
        for _ in range(rng.choice([1, 1, 1, 2, 3])):
            mutate(m)
        text = json.dumps(m)
        if rng.random() < 0.1:
            text = text[:rng.randrange(len(text))]
        with open(bad, "w") as f:
            f.write(text)
        try:
            eng.load_from_file(bad)
            eng.next_step(2)
        except RuntimeError:
            refused += 1
        eng.load_from_file(good)
        eng.next_step(1)
        assert eng.vehicle_count() == doc["activeVehicleCount"] or eng.vehicle_count() > 0
    assert refused > rounds // 2
    return refused
