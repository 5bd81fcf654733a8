"""One rank of the multi-GPU parity test (launched by tests/test_gpu_multi.py through torch.distributed.run, or by hand:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29517 \
        tests/shard_rank_main.py 30 60 1230 25 0.5 10 1 0.02

Every rank steps its strip of ONE simulation (peer-memory seam exchange, or NCCL send/recv with
CITYFLOW_B200_SHARD_TRANSPORT=nccl); the engine's COLLECTIVE observations -- get_vehicle_count() every 5 steps,
get_lane_vehicle_count() and get_lane_waiting_vehicle_count() every `every` steps -- are compared on rank 0 with the
unmodified reference (oracle/_ref/refdump counts, thread_num = host cores) on the same scenario, through its pinned results
(tests/refpin.py shard_runs)."""
import json
import os
import sys
import tempfile
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cityflow_b200  # noqa: E402
from cityflow_b200 import scenario  # noqa: E402
import refpin  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    a = sys.argv[1:]
    rows, cols, steps, every = int(a[0]), int(a[1]), int(a[2]), int(a[3])
    frac, interval, seed = float(a[4]), float(a[5]), int(a[6])
    spread = float(a[7]) if len(a) > 7 else 0.0
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    d = tempfile.mkdtemp()
    cfg = scenario.make_grid_scenario(d, rows, cols, dense=dict(frac=frac, interval=interval, seed=seed, fleet_spread=spread), name="sh")
    ref = None
    if rank == 0:
        ref = refpin.load("shard_runs")[refpin.shard_run_key(a)]
    dist.barrier()
    ids = [cityflow_b200.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    eng = cityflow_b200.Engine(cfg, thread_num=1, device=local, shard_rank=rank, shard_world=world, nccl_id=ids[0])
    lane_ids = eng.lane_ids()
    bad = []
    t_step = 0.0
    for s in range(1, steps + 1):
        t0 = time.perf_counter()
        eng.next_step()
        t_step += time.perf_counter() - t0
        if s % 5 == 0 or s == steps:
            n = eng.get_vehicle_count()                      # collective
            if ref is not None and n != ref["vehicle_count"][str(s)]:
                bad.append("step %d: vehicle count %d, reference %d" % (s, n, ref["vehicle_count"][str(s)]))
        if s % every == 0 or s == steps:
            lanes = eng.get_lane_vehicle_count()            # collective
            wait = eng.get_lane_waiting_vehicle_count()     # collective
            if ref is not None:
                want = ref["lanes"][str(s)]
                if refpin.lane_digest([lanes[k] for k in lane_ids]) != want["lane_count"]:
                    bad.append("step %d: lane counts differ" % s)
                if refpin.lane_digest([wait[k] for k in lane_ids]) != want["lane_waiting"]:
                    bad.append("step %d: lane waiting counts differ" % s)
        if len(bad) > 6:
            break
    t = torch.tensor([eng.tie_count(), len(bad)], device="cuda", dtype=torch.int64)
    dist.all_reduce(t)
    ties, nbad = int(t[0]), int(t[1])
    dist.barrier()
    if rank == 0:
        for b in bad[:8]:
            print(b)
        print("SHARD_PARITY " + json.dumps({"world": world, "grid": [rows, cols], "steps": steps, "equal": nbad == 0, "ties": ties,
                                           "transport": os.environ.get("CITYFLOW_B200_SHARD_TRANSPORT", "p2p"),
                                           "host_ms_per_step_enqueue": 1e3 * t_step / steps}), flush=True)
    del eng
    dist.destroy_process_group()
    sys.exit(0 if nbad == 0 else 1)


if __name__ == "__main__":
    main()
