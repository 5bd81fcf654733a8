"""The Python surface, object for object: the reference's own pybind11 module (oracle/_ref/cityflow*.so, the unmodified
reference) and whatever `import cityflow` resolves to -- this repository's module -- get the same calls (steps, RL phases,
push_vehicle, set_vehicle_speed, set_vehicle_route, set_random_seed, reset) and must return EQUAL Python objects from every
getter, every step: the dicts of get_lane_vehicle_count / get_lane_waiting_vehicle_count / get_vehicle_speed /
get_vehicle_distance (exact floats), the lists of get_vehicles (running and all) and of get_lane_vehicles (order on the
lane included), get_vehicle_info's string dict, get_leader, times, and the same exceptions.  TEST INFRASTRUCTURE.

The reference's side is pinned (tests/golden/reference/api_transcript.json, recorded by `tests/refpin.py api_transcript`):
a digest of every call's result (tests/refpin.py canonical(): numbers as the bits of a double) per ten steps.

Run as a script (`python tests/api_parity_main.py <config.json> <steps>`) it prints "OK ..." -- the CPU suite does that
in a child process whose PYTHONPATH puts the emulated-device build of the module first (tests/test_cpu.py); the GPU suite
calls compare_with_reference() in-process with the real module."""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GROUP = 10   # steps per pinned digest


def transcript(mod, cfg: str, steps: int):
    """Runs the script on a `mod.Engine`; yields (step, the result of every call made in that step, counters)."""
    eng = mod.Engine(cfg, thread_num=1)
    c = json.load(open(cfg))
    net = json.load(open(c["dir"] + c["roadnetFile"]))
    real = [i["id"] for i in net["intersections"] if not i["virtual"]]
    flows = json.load(open(c["dir"] + c["flowFile"]))
    some_route = flows[3]["route"]
    stats = dict(steps=0, infos=0, leaders=0, custom=0, rerouted_ok=0, rerouted_no=0, vehicles=0)
    out = []

    def call(name, *args, **kw):
        """the result, or the kind of exception (pybind maps std::runtime_error to RuntimeError in both modules)"""
        try:
            r = ("ok", getattr(eng, name)(*args, **kw))
        except Exception as ex:   # noqa: BLE001
            r = ("raised", type(ex).__name__)
        out.append((name, r))
        return r

    for s in range(1, steps + 1):
        stats["steps"] = s
        out = []
        if s % 10 == 1 and c.get("rlTrafficLight"):
            for k, i in enumerate(real):
                call("set_tl_phase", i, (s // 10 + k) % 8)
        if s in (40, 41, 150):
            call("push_vehicle", {"speed": 3.0, "length": 6.5, "maxSpeed": 12.0} if s != 41 else {}, some_route)
        if s == 120:
            call("set_random_seed", 77)
        if s == 200:
            call("reset", seed=False)
        running = call("get_vehicles")[1]
        if s % 25 == 3:
            for vid in running[:: max(1, len(running) // 5)]:
                call("set_vehicle_speed", vid, 0.5 * eng.get_vehicle_speed()[vid])
                stats["custom"] += 1
            call("set_vehicle_speed", "flow_999999_0", 1.0)     # unknown vehicle: raises
        if s % 30 == 7:
            for j, vid in enumerate(running[1:: max(1, len(running) // 9)]):
                target = flows[(s + j) % len(flows)]["route"][-1:] if j % 3 else ["no_such_road"]
                ok = call("set_vehicle_route", vid, target)[1]
                stats["rerouted_ok" if ok is True else "rerouted_no"] += 1
        call("next_step")
        assert call("get_vehicle_count")[1] == len(call("get_vehicles")[1])
        call("get_vehicles", include_waiting=True)
        call("get_current_time")
        call("get_lane_vehicle_count")
        call("get_lane_waiting_vehicle_count")
        call("get_lane_vehicles")
        call("get_vehicle_speed")
        call("get_vehicle_distance")
        call("get_average_travel_time")
        running = eng.get_vehicles()
        for vid in running[:: max(1, len(running) // 6)]:
            call("get_vehicle_info", vid)
            call("get_leader", vid)
            stats["infos"] += 1
        stats["vehicles"] = len(running)
        yield s, out, stats


def _digests(mod, cfg: str, steps: int):
    """(steps of the group, digest of its calls' results, counters) per GROUP steps"""
    import refpin
    assert steps % GROUP == 0, steps
    h = hashlib.sha256()
    for s, out, stats in transcript(mod, cfg, steps):
        h.update(refpin.canonical(out).encode())
        if s % GROUP == 0:
            yield [s - GROUP + 1, s], h.hexdigest()[:16], stats
            h = hashlib.sha256()


def record(ref_mod, cfg: str, steps: int) -> dict:
    return {"group": GROUP, "entries": [{"steps": a, "digest": d} for a, d, _ in _digests(ref_mod, cfg, steps)]}


def compare_with_reference(ours_mod, cfg: str, steps: int) -> dict:
    import refpin
    pin = refpin.load("api_transcript")
    assert pin["group"] == GROUP and steps <= GROUP * len(pin["entries"]), (steps, len(pin["entries"]))
    stats = None
    for (a, d, stats), want in zip(_digests(ours_mod, cfg, steps), pin["entries"]):
        assert a == want["steps"] and d == want["digest"], "steps %d..%d: some call returned another result than in the reference" % tuple(a)
    return dict(stats)


if __name__ == "__main__":
    import cityflow          # first: whatever PYTHONPATH puts first
    print("OK", json.dumps(compare_with_reference(cityflow, sys.argv[1], int(sys.argv[2]))), "with", cityflow.__file__)
