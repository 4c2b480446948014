#!/usr/bin/env python
"""Cost of the per-stream state calls: reset_streams, export_streams and import_streams of k streams out of --streams,
timed with CUDA events around each call (median of --reps after warm-up), next to a device-to-device copy of the same
payload bytes timed the same way and interleaved with them (the yardstick).  Also the time of resize_streams by one
stream (host clock around the synchronising call).

Bytes/s is payload bytes over time: export reads the state and writes the payload, import reads the payload and writes the
state, reset writes the state; the yardstick copy reads and writes the payload once.  Payloads of small k fit the 126 MB L2
of a B200; the k = --streams payload does not.  One JSON line per (workload, k), then one per workload for the resize;
the device name and power limit are part of every line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import continual_skeletons_b200 as cs  # noqa: E402

MODELS = {"cost_gcn": cs.CoStGcn, "cost_gcn_mod": cs.CoStGcnMod, "coa_gcn": cs.CoAGcn, "cos_tr": cs.CoSTr}


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return {"device": name, "power_limit": power}


def timed(fn):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    end.record()
    return start, end


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=4096)
    ap.add_argument("--ks", default="1,16,256,4096")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workloads", default=",".join(MODELS))
    ap.add_argument("--frames", type=int, default=12, help="frames stepped before timing, so the state is not all zero")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stream_state.py needs a CUDA device")
    info = device_info()
    dev = torch.device("cuda", 0)
    for tag in args.workloads.split(","):
        bench.set_geometry(tag)
        torch.manual_seed(0)
        model = MODELS[tag]({"dataset_name": bench.DATASET, "forward_mode": "frame", "time_chunk": 1})
        x = torch.rand((args.streams, bench.C_IN, bench.V, bench.S), device=dev)
        for _ in range(args.frames):
            model.forward_step(x)
        sb = model.stream_bytes()
        for k in [int(v) for v in args.ks.split(",")]:
            idx = [round(j * (args.streams - 1) / max(k - 1, 1)) for j in range(k)] if k > 1 else [args.streams // 2]
            state = model.export_streams(idx)
            src = torch.empty_like(state.payload)
            dst = torch.empty_like(state.payload)
            ops = {
                "reset": lambda: model.reset_streams(idx),
                "export": lambda: model.export_streams(idx),
                "import": lambda: model.import_streams(idx, state),
                "copy": lambda: dst.copy_(src),
            }
            times = {name: [] for name in ops}
            for rep in range(args.warmup + args.reps):
                events = {name: timed(fn) for name, fn in ops.items()}  # the four interleaved within every repetition
                torch.cuda.synchronize()
                if rep >= args.warmup:
                    for name, (s, e) in events.items():
                        times[name].append(s.elapsed_time(e))
            payload = k * sb
            line = dict(info, workload=tag, streams=args.streams, k=k, stream_bytes=sb, payload_bytes=payload, reps=args.reps)
            for name, ts in times.items():
                ms = statistics.median(ts)
                line[f"{name}_ms"] = round(ms, 5)
                line[f"{name}_GBps"] = round(payload / (ms * 1e-3) / 1e9, 1)
            for name in ("reset", "export", "import"):
                line[f"{name}_vs_copy"] = round(line["copy_ms"] / line[f"{name}_ms"], 3)
            print(json.dumps(line), flush=True)
        # resize by one stream, back and forth
        ts = []
        grow = list(range(args.streams)) + [-1]
        back = list(range(args.streams))
        for rep in range(1 + 5):
            torch.cuda.synchronize()
            s, e = timed(lambda: model.resize_streams(grow))
            torch.cuda.synchronize()
            if rep:
                ts.append(s.elapsed_time(e))
            model.resize_streams(back)
        print(json.dumps(dict(info, workload=tag, resize=f"{args.streams}->{args.streams + 1}",
                              resize_ms=round(statistics.median(ts), 3), state_bytes=model.state_bytes())), flush=True)
        model._engine.close()
        del model, state, src, dst
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
