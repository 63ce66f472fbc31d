"""gzip gRPC probe (not product): the grpc_h2 shape with every call gzip-compressed by the client — 256 connections x K unary calls per
step, 4 KiB text messages compressed at level 6 — through b2_h2_process_batch -> b2_h2_decompress_requests -> b2_h2_pack_responses
(echo of the inflated message, by reference).  Reports
  * the step: process + decompress + pack, host clock around calls that each end in a device synchronise;
  * the inflate kernels alone: CUDA events around k_h2_inflate (sizing pass, slot scan, writing pass) over every timed step;
msgs/s and inflated MB/s for both, with the card's name and power limit read in the same run.  Writes one JSON file."""
import argparse
import gzip
import json
import os
import random
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import brpc_b200  # noqa: E402
from brpc_b200.abi import H2_RESPONSE_DT  # noqa: E402
import _h2traffic as T  # noqa: E402
import _h2gzip as Z  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
        name, power = q.stdout.strip().split(",")[:2]
        return name.strip(), power.strip()
    except (OSError, ValueError):
        return "unknown", "unknown"


def make_steps(n_conns, k, n_steps, msg_bytes, seed):
    """the client bytes of every step (each connection: K complete calls, a connection WINDOW_UPDATE for the replies)"""
    rng = random.Random(seed)
    encs = [T.HpackEncoder(random.Random(seed + i)) for i in range(n_conns)]
    for e in encs:
        e.fixed_mode = "auto"                                    # a gRPC client's encoder: indexed once the fields are in the table
    sid = [1] * n_conns
    pool = [Z.text(rng, msg_bytes) for _ in range(64)]
    steps, n_in, n_out = [], 0, 0
    for s in range(n_steps):
        conn_bytes = []
        for i in range(n_conns):
            b = (T.PREFACE + T.settings()) if s == 0 else b""
            b += T.frame(8, 0, 0, (k * (msg_bytes + 5)).to_bytes(4, "big"))
            for _ in range(k):
                m = pool[rng.randrange(len(pool))]
                z = gzip.compress(m, compresslevel=6, mtime=0)
                b += Z.request(encs[i], sid[i], z, headers=[(b"grpc-encoding", b"gzip")])
                sid[i] += 2; n_in += len(z); n_out += len(m)
            conn_bytes.append(b)
        data, runs = brpc_b200.make_runs(conn_bytes)
        runs["socket_id"] = np.arange(n_conns, dtype=np.uint64)
        steps.append((data, runs))
    return steps, n_in / n_steps, n_out / n_steps


def one_step(ctx, data, runs, n_conns, k):
    rs, msgs, out = ctx.h2_process_batch(data, runs, msg_cap=n_conns * max(64, k), out_cap=n_conns * (64 << 10))
    res, _ = ctx.h2_decompress_requests(msgs, out_cap=16 << 20)
    st = ctx.stage_times()
    ct_off = 0
    r = np.zeros(len(msgs), H2_RESPONSE_DT)
    r["conn"] = msgs["run_idx"]; r["stream_id"] = msgs["stream_id"]; r["status_code"] = 200; r["flags"] = 1 | 16
    r["content_type_off"] = ct_off; r["content_type_len"] = 16
    r["body_off"] = res["out_off"]; r["body_len"] = res["out_len"]
    ctx.h2_pack_responses(np.frombuffer(b"application/grpc" + bytes(16), np.uint8), r)
    return len(msgs), res, st


def run(args, steps, per_out):
    ctx = brpc_b200.Context(device=0, max_batch_bytes=64 << 20, max_msgs=1 << 16, max_runs=args.conns, max_resp_bytes=64 << 20)
    ctx.h2_configure(max_conns=args.conns, max_pending=8, stream_bytes=69632)
    for i in range(args.conns):
        ctx.h2_conn_reset(i)
    for data, runs in steps[:args.warmup]:
        n, res, _ = one_step(ctx, data, runs, args.conns, args.k)
        assert n == args.conns * args.k and (res["status"] == Z.OK).all()
    kern_ms, n_msgs = 0.0, 0
    t0 = time.perf_counter()
    for data, runs in steps[args.warmup:]:
        n, res, st = one_step(ctx, data, runs, args.conns, args.k)
        kern_ms += sum(ms for name, ms in st)
        n_msgs += n
    wall = time.perf_counter() - t0
    assert (res["status"] == Z.OK).all()
    n_steps = len(steps) - args.warmup
    return {"steps": n_steps, "msgs": n_msgs,
            "step_ms": 1e3 * wall / n_steps, "msgs_per_s": n_msgs / wall, "inflated_MB_per_s": per_out * n_steps / wall / 1e6,
            "inflate_kernels_ms_per_step": kern_ms / n_steps, "inflate_kernels_msgs_per_s": n_msgs / (kern_ms / 1e3),
            "inflate_kernels_inflated_MB_per_s": per_out * n_steps / (kern_ms / 1e3) / 1e6,
            "stages_last_step_ms": {name: ms for name, ms in st}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--conns", type=int, default=256)
    ap.add_argument("--k", type=int, default=8, help="calls per connection and step")
    ap.add_argument("--msg-bytes", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "h2_gzip_probe.json"))
    args = ap.parse_args()
    name, power = card()
    steps, per_in, per_out = make_steps(args.conns, args.k, args.warmup + args.steps, args.msg_bytes, seed=7)
    results = []
    for rep in range(2):                                         # twice: the spread between repeats (the host is shared)
        r = run(args, steps, per_out); r["rep"] = rep
        results.append(r)
        print(json.dumps(r))
    doc = {"card": name, "power_limit": power, "workload": {"connections": args.conns, "calls_per_connection_per_step": args.k,
           "message_bytes": args.msg_bytes, "gzip_level": 6, "compressed_bytes_per_step": per_in, "inflated_bytes_per_step": per_out},
           "results": results}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print("card %s, power limit %s -> %s" % (name, power, args.out))


if __name__ == "__main__":
    main()
