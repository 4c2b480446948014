#!/usr/bin/env python
"""Cost of prime_streams: k joining streams primed from H = receptive_field frames of history on a handle of --streams
streams, timed with CUDA events around each call (the call ends in a device synchronise; median of --reps after warm-up).
The yardstick is forward_steps of the same H frames on a handle of k streams, with the same time chunk, timed the same
way and interleaved with the priming calls (its state is reset outside the timed region).  Also the kernel launches of one
call of each.

prime_streams walks the k streams' history on scratch state of its own (allocated, zeroed and freed within the call),
then gathers it into a payload and scatters that into the handle: the difference to the yardstick is that overhead.  One
JSON line per (workload, k); the device name and power limit are part of every line.
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import bench  # noqa: E402
import continual_skeletons_b200 as cs  # noqa: E402
from bench_stream_state import MODELS, device_info, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=4096)
    ap.add_argument("--ks", default="1,64,1024")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default=",".join(MODELS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_prime_streams.py needs a CUDA device")
    info = device_info()
    dev = torch.device("cuda", 0)
    for tag in args.workloads.split(","):
        bench.set_geometry(tag)
        torch.manual_seed(0)
        hp = {"dataset_name": bench.DATASET, "forward_mode": "frame"}
        model = MODELS[tag](hp)
        H = model.receptive_field
        x = torch.rand((args.streams, bench.C_IN, bench.V, bench.S), device=dev)
        for _ in range(H):  # every stream past the receptive field: the handle at a steady frame count
            model.forward_step(x)
        for k in [int(v) for v in args.ks.split(",")]:
            idx = [round(j * (args.streams - 1) / max(k - 1, 1)) for j in range(k)] if k > 1 else [args.streams // 2]
            clip = torch.rand((k, bench.C_IN, H, bench.V, bench.S), device=dev)
            yard = MODELS[tag](hp)
            yard.load_state_dict(model.state_dict())
            yard.forward_steps(clip)  # creates its state with the time chunk prime_streams picks for (k, H)
            tc, prime_tc = yard._engine.time_chunk, model._pick_time_chunk(k, H)
            n0 = model.launch_count()
            model.prime_streams(idx, clip)
            prime_launches = model.launch_count() - n0
            yard.clean_state()
            n0 = yard.launch_count()
            yard.forward_steps(clip)
            steps_launches = yard.launch_count() - n0
            times = {"prime": [], "steps": []}
            for rep in range(args.warmup + args.reps):
                yard.clean_state()
                torch.cuda.synchronize()
                events = {"prime": timed(lambda: model.prime_streams(idx, clip)), "steps": timed(lambda: yard.forward_steps(clip))}
                torch.cuda.synchronize()
                if rep >= args.warmup:
                    for name, (s, e) in events.items():
                        times[name].append(s.elapsed_time(e))
            line = dict(info, workload=tag, streams=args.streams, k=k, H=H, prime_time_chunk=prime_tc, steps_time_chunk=tc, reps=args.reps,
                        prime_launches=prime_launches, steps_launches=steps_launches)
            for name, ts in times.items():
                line[f"{name}_ms"] = round(statistics.median(ts), 3)
            line["prime_vs_steps"] = round(line["prime_ms"] / line["steps_ms"], 3)
            print(json.dumps(line), flush=True)
            yard._engine.close()
            del yard, clip
            torch.cuda.empty_cache()
        model._engine.close()
        del model
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
