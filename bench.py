#!/usr/bin/env python
"""bench.py — echo QPS of the B200 brpc hot path (BASELINE.json metric).

Workload (config.workload): BASELINE configs[1] — example/multi_threaded_echo_c++ shape:
64 client connections per GPU, baidu_std, 1 KB 'r' payload (client.cpp:116), every
connection's read buffer holding RUN_MIB MiB of pipelined requests whose last frame
is cut mid-way.  One *step* = one pass of the whole hot path over one such batch
(cut loop -> RpcMeta decode -> echo -> response pack), 256 MiB in / ~249 MiB out at
N=1, i.e. larger than the 126 MB L2, so no L2 flush is needed between iterations.

  value    : messages/s with the batch resident in HBM (kernel pipeline only)
  e2e      : messages/s through b2_process_batch with PINNED HOST buffers, H2D of the
             request bytes and D2H of descriptors + response bytes inside the timed region
  roofline : dominant kernel (k_pack) algorithmic bytes / CUDA-event time vs measured HBM peak
  cpu_baseline : the oracle port (oracle/liboracle.so) on the host cores, bounded sample

`--impl reference` times the CPU implementation of the same path on all host threads
(the reference itself cannot be built: SURVEY §0 — protoc/libprotobuf/gflags absent).
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

PAYLOAD = 1024
N_SOCKETS = 64
DESC_BYTES = 64


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill(); out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [x for x in sm if x > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def pin_to_gpu_numa(gpu_index):
    """Run this rank (and allocate its pinned buffers) on the CPUs next to its GPU: with 8 ranks the host<->device copies of
    the e2e leg otherwise cross the socket interconnect (SURVEY §8e: one pinned pool per NUMA node)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = [64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1 and 64 * w + b < n_cpu]
        if cpus:
            os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return 0


def ncu_traffic(kernel, args):
    """dram bytes read + written per launch of `kernel` from the committed `ncu --set full` capture of this same workload
    (profiles/r2_ncu_summary.json; it names the kernels it saw, so a renamed / restructured kernel reads as None rather
    than as a stale number), or None when the capture does not cover the configuration being run."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_ncu_summary.json")) as f:
            cap = json.load(f)
        w = cap["workload"]
        if (w["payload_bytes"], w["run_mib"], w["connections"]) != (args.payload, args.run_mib, N_SOCKETS) or args.checksum or args.payload_kind:
            return None
        ks = {n.replace("void ", "").split("<")[0].strip(): v for n, v in cap["kernels"].items()}
        k = ks.get(kernel) or ks.get(kernel + "_tma")
        return None if k is None else (k["dram_read_MB"] + k["dram_write_MB"]) * 1e6
    except Exception:
        return None


def build_batch(run_mib, rank, pinned=True, payload=PAYLOAD, checksum=0, kind=0):
    from brpc_b200 import press
    from brpc_b200.abi import PinnedBuffer
    run_bytes = int(run_mib * (1 << 20)) - 16 * 7          # not a multiple of the frame: every run ends mid-frame
    stride = (run_bytes + 15) // 16 * 16
    nbytes = N_SOCKETS * stride
    buf = PinnedBuffer(nbytes) if pinned else None
    data = buf.array if pinned else np.zeros(nbytes, np.uint8)
    sp = press.spec(payload_bytes=payload, payload_kind=kind, checksum_type=checksum)
    # sockets are sharded over GPUs by socket id (SURVEY §8e): rank r serves ids r*64 .. r*64+63
    runs, n_full = press.fill_batch(sp, data, N_SOCKETS, run_bytes, start_index=rank * 1000003)
    runs["socket_id"] += rank * N_SOCKETS
    return buf, data, runs, n_full, nbytes


def cpu_arm(data, runs, threads, min_seconds):
    """Time the oracle port over `runs` with `threads` host threads (ctypes drops the GIL).
    The cut loop is serial per connection, but brpc hands every cut message to its own bthread
    (input_messenger.cpp:272), so to let the CPU use all its cores each run is first split at
    frame boundaries (found by one untimed oracle pass) into enough sub-runs to feed every thread."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _oracle as O
    cfg = O.make_config()
    if threads > len(runs):
        rs0, m0, _ = O.process_batch(cfg, data, runs)
        pieces = max(1, (2 * threads + len(runs) - 1) // len(runs))
        sub = []
        for r in range(len(runs)):
            a, n = int(rs0["first_msg"][r]), int(rs0["n_msgs"][r])
            offs = m0["frame_off"][a:a + n].astype(np.int64)
            end = int(runs["offset"][r]) + int(runs["length"][r])
            cuts = [int(offs[k * n // pieces]) for k in range(pieces)] if n >= pieces else [int(runs["offset"][r])]
            cuts[0] = int(runs["offset"][r])
            for k, c in enumerate(cuts):
                e = cuts[k + 1] if k + 1 < len(cuts) else end
                sub.append((int(runs["socket_id"][r]), c, e - c, -1, 0))
        runs = np.array(sub, dtype=runs.dtype)
    parts = [p for p in np.array_split(np.arange(len(runs)), threads) if len(p)]
    bufs = []
    for p in parts:
        sub = np.ascontiguousarray(runs[p])
        nb = int(sub["length"].sum())
        bufs.append((sub, np.zeros(len(p), O.RUN_STATUS_DT), np.zeros(nb // 1000 + 64, O.MSG_DT),
                     np.zeros(nb + (1 << 16), np.uint8), C.c_uint32(), C.c_uint32()))

    def work(b):
        sub, rs, msgs, resp, nm, rb = b
        rc = O.lib.orc_process_batch(C.byref(cfg), data.ctypes.data, data.nbytes, sub.ctypes.data, len(sub), rs.ctypes.data,
                                     msgs.ctypes.data, len(msgs), C.byref(nm), resp.ctypes.data, len(resp), C.byref(rb))
        assert rc == 0

    # persistent worker threads (ctypes drops the GIL inside the oracle call); every pass runs each worker's share `reps`
    # times so that thread wake-up costs stay small against the work being timed
    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(max_workers=len(bufs))
    reps = 4 if len(bufs) > 1 else 1

    def work_reps(b):
        for _ in range(reps):
            work(b)

    def one_pass():
        t0 = time.perf_counter()
        list(pool.map(work_reps, bufs))
        dt = time.perf_counter() - t0
        return dt, reps * sum(b[4].value for b in bufs)

    one_pass()                                    # warm-up: page faults, tables, thread start
    best, n, spent = None, 0, 0.0
    while spent < min_seconds or n < 3:
        dt, msgs = one_pass()
        spent += dt; n += 1
        if best is None or dt < best[0]:
            best = (dt, msgs)
    pool.shutdown()
    return best[1] / best[0], best[1], n


def grpc_h2_main(args):
    """BASELINE configs[3]: h2/gRPC unary calls with 4 KB messages, 256 connections per GPU, through the h2 entry points
    of the C ABI (b2_h2_process_batch + b2_h2_pack_responses, host buffers, synchronous): parse + echo + reply framing.
    A side measurement (the h2 path is one thread per connection; it is latency-, not bandwidth-bound)."""
    import torch
    import brpc_b200
    from brpc_b200.abi import H2_RESPONSE_DT
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _h2traffic as T
    import random
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    dev = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(dev)
    use_dist = world > 1
    if use_dist:                                                # one process per GPU, connections sharded by rank: no exchange step
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    pin_to_gpu_numa(dev)
    hbm_peak, peak_src = read_peaks()
    n_conns, K, msg_len = 256, args.frames_per_stream, args.payload if args.payload != 1024 else 4096
    steps, warmup = max(1, args.steps), max(3, args.warmup)
    rng = random.Random(20260921 + rank)
    ctx = brpc_b200.Context(device=dev, max_batch_bytes=64 << 20, max_msgs=1 << 16, max_runs=1024, max_resp_bytes=128 << 20)
    message = bytes(rng.choice(b"abcdefghijklmnopqrstuvwxyz0123456789") for _ in range(msg_len))
    # one batch = K complete calls per connection; the same bytes are replayed every step with fresh (growing) stream ids
    first_batch, batch, sid_pos = [], [], []
    for cidx in range(n_conns):
        ctx.h2_conn_reset(cidx)
        enc = T.HpackEncoder(rng); enc.fixed_mode = "auto"              # indexed when present, else literal + incremental indexing
        warm = b"".join(T.request_frames(rng, enc, 1, message=message, chunk=16384))       # fills the HPACK tables: later calls are all table hits
        first_batch.append(T.PREFACE + T.settings() + warm)
        calls = [T.request_frames(rng, enc, 3 + 2 * k, message=message, chunk=16384) for k in range(K)]
        # the client returns the connection-level credit the replies of the previous round used (WINDOW_UPDATE on stream 0)
        batch.append(T.frame(8, 0, 0, (K * (msg_len + 16)).to_bytes(4, "big")) + b"".join(b"".join(c) for c in calls))
    data0, runs0 = brpc_b200.make_runs(first_batch)
    rs, msgs, out = ctx.h2_process_batch(data0, runs0)
    assert int(rs["n_msgs"].sum()) == n_conns
    data_, runs = brpc_b200.make_runs(batch)
    from brpc_b200.abi import PinnedBuffer
    pin_in = PinnedBuffer(len(data_)); data = pin_in.array; data[:] = data_        # host buffers are pinned, like IOBuf blocks from b2_block_alloc
    pin_out = PinnedBuffer(n_conns * (K * 1024 + 8192)); pin_pack = PinnedBuffer(n_conns * K * (msg_len + 256) + 4096)
    pos = []                                                   # offsets of every frame's stream-id field
    for r_ in runs:
        p_ = int(r_["offset"]); end = p_ + int(r_["length"])
        while p_ < end:
            ln = (int(data[p_]) << 16) | (int(data[p_ + 1]) << 8) | int(data[p_ + 2])
            pos.append(p_ + 5); p_ += 9 + ln
    pos = np.array(pos, dtype=np.int64)
    pos = pos[(data[pos] | data[pos + 1] | data[pos + 2] | data[pos + 3]) != 0]        # stream 0 (connection) frames keep their id
    base_sid = ((data[pos].astype(np.int64) << 24) | (data[pos + 1].astype(np.int64) << 16) | (data[pos + 2].astype(np.int64) << 8) | data[pos + 3])

    def set_round(t):
        sid = base_sid + 2 * K * t
        data[pos] = (sid >> 24) & 255; data[pos + 1] = (sid >> 16) & 255; data[pos + 2] = (sid >> 8) & 255; data[pos + 3] = sid & 255

    ct = b"application/grpc"
    # where the content-type value sits inside a request's header records (same for every steady-state call)
    hb0 = bytes(out[msgs[0]["headers_off"]:msgs[0]["headers_off"] + msgs[0]["headers_len"]]); ct_rel = hb0.index(ct)
    def one_step(t, check=False):
        set_round(t)
        rs, msgs, out = ctx.h2_process_batch(data, runs, msg_cap=n_conns * (K + 2), out=pin_out.array)
        n = len(msgs)
        assert n == n_conns * K, (n, rs["parse_error"][:4])
        # echo: the reply message is the request message, still on the device (input buffer when one DATA frame carried it,
        # else the out buffer); the reply's content-type is the request's own value inside out — nothing is uploaded again
        resps = np.zeros(n, dtype=H2_RESPONSE_DT)
        resps["conn"] = runs["socket_id"][msgs["run_idx"]]; resps["stream_id"] = msgs["stream_id"]; resps["status_code"] = 200
        resps["flags"] = 1 | 8 | np.where(msgs["flags"] & 16, 2, 4)
        resps["content_type_off"] = msgs["headers_off"] + ct_rel; resps["content_type_len"] = len(ct)
        resps["body_off"] = msgs["msg_off"]; resps["body_len"] = msgs["msg_len"]
        pout, poffs, plens = ctx.h2_pack_responses(None, resps, raw=True, out=pin_pack.array)
        if check:
            assert np.all(plens > msg_len) and bytes(pout[poffs[0] + 9:poffs[0] + 10]) == b"\x88"       # HEADERS begin with :status 200 (static index 8)
        return n
    for t in range(warmup):
        one_step(t, check=True)
    sampler = ClockSampler(dev); sampler.start()
    if use_dist:
        dist.barrier()
    torch.cuda.synchronize(); t0 = time.perf_counter(); total = 0
    for t in range(steps):
        total += one_step(warmup + t)
    torch.cuda.synchronize()
    if use_dist:
        dist.barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    if use_dist:                                                # max time over ranks, summed calls; the bvar-like counters go through NCCL too
        tw = torch.tensor([wall], dtype=torch.float64, device="cuda"); dist.all_reduce(tw, op=dist.ReduceOp.MAX); wall = tw.item()
        tt = torch.tensor([float(total)], dtype=torch.float64, device="cuda"); dist.all_reduce(tt, op=dist.ReduceOp.SUM); total = tt.item()
    ms = wall * 1e3 / steps
    if rank == 0:
        line = {"metric": "h2/gRPC echo QPS, %d B messages" % msg_len, "value": total / wall, "unit": "msgs/s", "n_gpus": world if use_dist else 1, "steps": steps, "warmup": warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": "grpc_c++-style unary calls over h2: %d connections/GPU x %d calls per batch, %d B messages, HPACK dynamic-table hits" % (n_conns, K, msg_len),
                           "note": "timed through the synchronous C ABI with host buffers (copies and the Python glue that builds the response list included)"},
                "e2e": {"value": total / wall, "unit": "msgs/s", "h2d_bytes_per_step": int(data.nbytes + runs.nbytes + n_conns * K * 48),
                        "d2h_bytes_per_step": int(n_conns * K * (64 + 320 + msg_len + 64) + n_conns * 32)},
                "gpu_launches": int(2 * steps), "clocks": clocks}
        if not args.no_cpu_baseline:
            import _oracle as O
            conns = [O.H2Conn() for _ in range(8)]
            for i_, c_ in enumerate(conns): c_.consume(first_batch[i_])
            t1 = time.perf_counter(); n = 0; rounds = 0
            while time.perf_counter() - t1 < 5.0:
                set_round(1000 + rounds); rounds += 1
                for i_, c_ in enumerate(conns):
                    o_, l_ = int(runs["offset"][i_]), int(runs["length"][i_])
                    e_, cons_, om, _, ob, _, _ = c_.consume(data[o_:o_ + l_].tobytes())
                    for m_ in om:
                        c_.pack_response(int(m_["stream_id"]), bytes(ob[m_["msg_off"]:m_["msg_off"] + m_["msg_len"]])); n += 1
            line["cpu_baseline"] = {"value": n / (time.perf_counter() - t1), "unit": "msgs/s", "cores": 1, "kind": "port",
                                    "sample": "8 of the %d connections, parse + pack through the oracle (Python glue included), ~5 s" % n_conns}
        print(json.dumps(line))
    if use_dist:
        dist.destroy_process_group()
    return 0


def stream_snappy_main(args):
    """BASELINE configs[4]: streaming_rpc DATA frames carrying 256 KiB snappy-compressed messages, 64 streams per GPU;
    the device cuts the frames, decodes StreamFrameMeta and decompresses every payload (b2_set_stream_handler).
    Same JSON shape as the headline line; the unit of work is one frame."""
    import torch
    import brpc_b200
    from brpc_b200 import press
    from brpc_b200.abi import PinnedBuffer
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    use_dist = world > 1
    if use_dist:
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = local_rank if use_dist else 0
    torch.cuda.set_device(dev)
    hbm_peak, peak_src = read_peaks()
    steps, warmup = max(1, args.steps), max(3, args.warmup)
    RAW = 256 << 10
    rng = np.random.default_rng(20260921 + rank)
    table = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ", np.uint8)
    pattern = np.resize(table[:36], RAW)                                   # brpc_snappy_compress_unittest.cpp text: a-z0-9 repeating
    if args.payload_kind == 0:
        raws = [pattern]
    else:
        raws = [table[rng.integers(0, 62, RAW)] for _ in range(4)]         # uniform random over the 62-symbol table
    K = args.frames_per_stream
    n_frames = N_SOCKETS * K
    gen = brpc_b200.Context(device=dev, max_batch_bytes=8 << 20, max_msgs=64, max_runs=8)
    flat = np.concatenate(raws)
    comps = gen.snappy_compress_batch(flat, np.arange(len(raws), dtype=np.uint32) * RAW, np.full(len(raws), RAW, np.uint32),
                                      len(raws) * (RAW + RAW // 6 + 64))  # the device encoder (bit-exact with the vendored snappy)
    del gen
    streams = []
    for s_ in range(N_SOCKETS):
        sid = rank * N_SOCKETS + s_
        streams.append(b"".join(press.stream_frame(1000 + sid, 5000 + sid, comps[(s_ + i) % len(comps)]) for i in range(K)))
    stride = (max(len(x) for x in streams) + 15) // 16 * 16
    nbytes = N_SOCKETS * stride
    buf = PinnedBuffer(nbytes)
    runs = np.zeros(N_SOCKETS, dtype=brpc_b200.RUN_DT)
    for s_, x in enumerate(streams):
        buf.array[s_ * stride:s_ * stride + len(x)] = np.frombuffer(x, np.uint8)
        runs[s_] = (rank * N_SOCKETS + s_, s_ * stride, len(x), -1, 0)
    out_bytes = n_frames * (RAW + 64) + (4 << 20)
    mk = lambda: brpc_b200.Context(device=dev, max_batch_bytes=nbytes + (1 << 20), max_msgs=n_frames + 1024, max_runs=N_SOCKETS,
                                   max_resp_bytes=out_bytes, stream_handler=1)
    ctxs = [mk() for _ in range(2)]
    rs, msgs, resp, info = ctxs[0].process_batch_ptr(buf.ptr, nbytes, runs)
    assert len(msgs) == n_frames and np.all(msgs["status"] == 4) and np.all(msgs["resp_len"] == RAW) and np.all(msgs["error_code"] == 0)
    for i in range(0, n_frames, max(1, n_frames // 16)):                  # decompressed bytes == what was compressed
        s_, k = divmod(i, K)
        o = int(msgs["resp_off"][i])
        assert np.array_equal(resp[o:o + RAW], raws[(s_ + k) % len(raws)]), "stream frame %d decompressed wrong" % i
    req_bytes = int(rs["consumed"].sum())

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()
    for cx in ctxs:
        cx.upload_ptr(buf.ptr, nbytes, runs)
    for s_ in range(warmup * 2):
        ctxs[s_ % 2].launch()
    for cx in ctxs:
        cx.wait()
    sampler = ClockSampler(dev); sampler.start()
    barrier()
    for s_ in range(steps):
        ctxs[s_ % 2].launch()
    for cx in ctxs:
        cx.wait()
    barrier()
    clocks = sampler.stop()
    dev_ms = max(ctxs[0].elapsed_ms_to(cx) for cx in ctxs[:min(2, steps)])
    stage_acc = {}
    for _ in range(3):
        ctxs[0].execute()
        for name, ms in ctxs[0].stage_times():
            stage_acc.setdefault(name, []).append(ms)
    stages = {k: statistics.mean(v) for k, v in stage_acc.items()}
    e2e_steps = max(4, min(steps, 12))
    for cx in ctxs:
        cx.submit_ptr(buf.ptr, nbytes, runs)
    for cx in ctxs:
        cx.collect()
    barrier()
    t0 = time.perf_counter()
    for s_ in range(min(2, e2e_steps)):
        ctxs[s_].submit_ptr(buf.ptr, nbytes, runs)
    for s_ in range(e2e_steps):
        cx = ctxs[s_ % 2]
        r3, m3, p3, _ = cx.collect()
        assert len(m3) == n_frames
        if s_ + 2 < e2e_steps:
            cx.submit_ptr(buf.ptr, nbytes, runs)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    t_dev = torch.tensor([dev_ms, e2e_ms], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(n_frames)], dtype=torch.float64, device="cuda")
    counters = ctxs[0].counters()
    if use_dist:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX); dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        cnt = torch.tensor(counters, dtype=torch.int64, device="cuda")
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)                        # the NCCL counter reduce of configs[4]
        counters = cnt.tolist()
    dev_ms_max, e2e_ms_max = t_dev.tolist()
    ms_per_step = dev_ms_max / steps
    if rank == 0:
        alg = float(req_bytes + n_frames * (RAW + DESC_BYTES))            # SURVEY §8d: 12+meta+C read, U written, 64 B desc
        dom = max(stages, key=stages.get)
        line = {"metric": "streaming_rpc snappy frames (256 KiB) decompressed", "value": tot.item() / (ms_per_step * 1e-3), "unit": "frames/s",
                "n_gpus": world if use_dist else 1, "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": "streaming_echo_c++-style STRM DATA frames, %d streams/GPU x %d frames, 256 KiB %s messages, snappy"
                                       % (N_SOCKETS, K, "a-z0-9 pattern" if args.payload_kind == 0 else "random-62"),
                           "compressed_bytes_per_frame": len(comps[0]), "l2": "outputs larger than L2"},
                "decompressed_GBps": tot.item() * RAW / (ms_per_step * 1e-3) / 1e9,
                "e2e": {"value": tot.item() / (e2e_ms_max * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": int(nbytes + runs.nbytes),
                        "d2h_bytes_per_step": int(n_frames * (RAW + 64) + len(rs) * 32), "ms_per_step": e2e_ms_max},
                "gpu_launches": int(steps * info["n_launches"]),
                "roofline": {"bound": "hbm", "kernel": "k_" + dom, "achieved": alg / (stages[dom] * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": alg / (stages[dom] * 1e-3) / 1e9 / hbm_peak, "traffic": None, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg, "kernel_ms": stages[dom], "stage_ms": stages},
                "clocks": clocks, "counters_allreduced": counters}
        if not args.no_cpu_baseline:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import _oracle as O
            cfg = O.make_config(stream_handler=1)
            sub = runs[:4].copy()
            t0 = time.perf_counter(); n = 0; best = None
            while time.perf_counter() - t0 < 8.0 or n < 2:
                t1 = time.perf_counter()
                ors, om, _ = O.process_batch(cfg, buf.array, sub, msg_cap=4 * K + 16, resp_cap=4 * K * (RAW + 64) + (1 << 20))
                dt = time.perf_counter() - t1; n += 1
                best = dt if best is None or dt < best else best
            line["cpu_baseline"] = {"value": len(om) / best, "unit": "frames/s", "cores": 1, "kind": "port",
                                    "sample": "4 of the %d streams (%d frames/pass), best of %d passes, single thread" % (N_SOCKETS, len(om), n)}
        print(json.dumps(line))
    if use_dist:
        dist.destroy_process_group()
    return 0


def load_press():
    """tools/libb2press.so (the rpc_press-like traffic source, host code) without importing the product package."""
    class Spec(C.Structure):
        _fields_ = [("service", C.c_char_p), ("method", C.c_char_p), ("payload_bytes", C.c_uint32), ("attachment_bytes", C.c_uint32),
                    ("payload_kind", C.c_int32), ("checksum_type", C.c_int32), ("seed", C.c_uint64)]
    so = os.path.join(ROOT, "brpc_b200", "tools", "libb2press.so")
    if not os.path.exists(so):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, os.path.join(ROOT, "brpc_b200", "tools", "rpc_press.cpp")])
    lib = C.CDLL(so)
    lib.b2press_fill_run.restype = C.c_uint64
    lib.b2press_fill_run.argtypes = [C.POINTER(Spec), C.POINTER(C.c_uint64), C.c_void_p, C.c_size_t]
    return lib, Spec


RUN_DT = np.dtype([("socket_id", "<u8"), ("offset", "<u4"), ("length", "<u4"), ("preferred_proto", "<i4"), ("flags", "<u4")])


def socket_ids_of(rank, world):
    """The connections rank `rank` serves: gpu = SlotOfVRefId(socket_id) % n_gpus (SURVEY §8e; brpc_b200/shard.py:owner_of)."""
    ids = np.arange(N_SOCKETS * max(1, world), dtype=np.uint64)
    own = (ids & np.uint64(0xffffffff)) % np.uint64(max(1, world))
    return ids[own == rank]


def fill_batch_plain(data, run_mib, rank, world, payload=PAYLOAD, checksum=0, kind=0):
    lib, Spec = load_press()
    run_bytes = int(run_mib * (1 << 20)) - 16 * 7
    stride = (run_bytes + 15) // 16 * 16
    sp = Spec(b"example.EchoService", b"Echo", payload, 0, kind, checksum, 20260921)
    ids = socket_ids_of(rank, world)
    runs = np.zeros(N_SOCKETS, dtype=RUN_DT)
    total = 0
    for s_ in range(N_SOCKETS):
        idx = C.c_uint64((int(ids[s_]) << 32) + 1000003 * rank)
        total += lib.b2press_fill_run(C.byref(sp), C.byref(idx), data.ctypes.data + s_ * stride, run_bytes)
        runs[s_] = (int(ids[s_]), s_ * stride, run_bytes, -1, 0)
    return runs, int(total), N_SOCKETS * stride


def dump_outputs(out_dir, rs, msgs, resp, sample=4096, reply_bytes=2048):
    """What a caller of the timed path receives for the batch, as float64 / float32 .npy files: per connection, run_<field>
    and the zlib CRC-32s of all its message descriptors (run_msgs_crc32) and of its replies in order (run_reply_crc32); msg_index, a
    fixed seeded sample of `sample` messages, with msg_<field> their descriptors and reply_bytes / reply_bytes_off the first
    `reply_bytes` bytes of their replies, concatenated.  Every value is exact: the 64-bit ids rpc_press.cpp writes stay
    below 2^53."""
    import zlib
    os.makedirs(out_dir, exist_ok=True)
    save = lambda name, a, dt=np.float64: np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a).astype(dt))
    for f in rs.dtype.names:
        save("run_" + f, rs[f])
    resp = np.asarray(resp)
    save("run_msgs_crc32", [zlib.crc32(msgs[int(r["first_msg"]):int(r["first_msg"]) + int(r["n_msgs"])].tobytes()) for r in rs])
    offs, lens = msgs["resp_off"].astype(np.int64), msgs["resp_len"].astype(np.int64)
    crc = np.zeros(len(rs), np.uint32)
    for r, o, n in zip(msgs["run_idx"], offs, lens):
        crc[r] = zlib.crc32(resp[o:o + n], int(crc[r]))
    save("run_reply_crc32", crc)
    idx = np.sort(np.random.default_rng(20260921).choice(len(msgs), min(sample, len(msgs)), replace=False))
    save("msg_index", idx)
    for f in msgs.dtype.names:
        save("msg_" + f, msgs[f][idx])
    parts = [resp[o:o + min(n, reply_bytes)] for o, n in zip(offs[idx], lens[idx])]
    save("reply_bytes", np.concatenate(parts) if parts else np.zeros(0, np.uint8), np.float32)
    save("reply_bytes_off", np.cumsum([0] + [len(p) for p in parts]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--run-mib", type=float, default=4, help="MiB pending per connection per batch (a fraction for many small connections)")
    ap.add_argument("--sockets", type=int, default=64, help="connections per GPU in one batch (the rpc_press sweep of BASELINE configs[2] uses 1024)")
    ap.add_argument("--tile", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--payload", type=int, default=1024, help="EchoRequest.message bytes (rpc_press sweep: 64..65536)")
    ap.add_argument("--checksum", type=int, default=0, help="1 = CRC32C on requests (-enable_checksum)")
    ap.add_argument("--payload-kind", type=int, default=0, help="0 = 'r' fill, 1 = random over 62 symbols")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--pipeline", type=int, default=2, help="resident batches in flight per GPU (one ctx + stream each)")
    ap.add_argument("--workload", default="echo", choices=["echo", "stream_snappy", "grpc_h2"],
                    help="echo = the headline metric; stream_snappy = BASELINE configs[4] (256 KiB snappy streaming frames), grpc_h2 = configs[3]")
    ap.add_argument("--frames-per-stream", type=int, default=8)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy (echo workload)")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "echo" or args.impl != "b200"):
        ap.error("--dump-outputs covers the echo workload of the b200 implementation")
    global N_SOCKETS
    N_SOCKETS = max(1, args.sockets)
    if args.run_mib == int(args.run_mib):
        args.run_mib = int(args.run_mib)
    if args.workload == "stream_snappy":
        return stream_snappy_main(args)
    if args.workload == "grpc_h2":
        return grpc_h2_main(args)
    steps, warmup = max(1, args.steps), max(3, args.warmup)
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    hbm_peak, peak_src = read_peaks()
    ncores = os.cpu_count() or 1
    workload = ("multi_threaded_echo_c++ baidu_std %d B payload: %d connections/GPU x %s MiB pending, runs cut mid-frame; batch %d MiB > L2 (no flush needed)"
                % (args.payload, N_SOCKETS, args.run_mib, int(N_SOCKETS * args.run_mib)))
    config = {"workload": workload, "payload_bytes": args.payload, "request_checksum": args.checksum, "connections_per_gpu": N_SOCKETS,
              "run_mib": args.run_mib, "l2": "inputs larger than L2", "pipeline_depth": args.pipeline,
              "sharding": "gpu = (socket_id & 0xffffffff) %% %d (shard.owner_of)" % max(1, world),
              "host": "each rank pinned to its GPU's NUMA node"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        nb = N_SOCKETS * ((int(args.run_mib * (1 << 20)) - 112 + 15) // 16 * 16)
        data = np.zeros(nb, np.uint8)
        runs, n_full, nbytes = fill_batch_plain(data, args.run_mib, 0, 1, payload=args.payload, checksum=args.checksum, kind=args.payload_kind)
        t0 = time.perf_counter()
        qps, msgs, passes = cpu_arm(data, runs, ncores, min_seconds=min(20.0, 1.0 * steps))
        config["reference_arm"] = ("oracle port of the reference path on %d host threads; every connection is split at frame boundaries by an UNTIMED pass so that all "
                                   "threads have work (brpc hands each cut message to its own bthread); brpc itself cannot be built here" % ncores)
        line = {"impl": "reference", "metric": "echo QPS, 1 KB baidu_std", "value": qps, "unit": "msgs/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * msgs / qps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": qps, "unit": "msgs/s", "cores": ncores, "kind": "port",
                                 "sample": "%d connections x %d MiB (%d msgs/pass) split at frame boundaries over the threads, "
                                           "best of %d passes, %d threads; oracle port of the reference path (brpc itself cannot be built here)"
                                           % (N_SOCKETS, args.run_mib, msgs, passes, ncores)},
                "e2e": {"value": qps, "unit": "msgs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "wall_s": time.perf_counter() - t0}
        print(json.dumps(line))
        return 0

    import torch
    import brpc_b200
    from brpc_b200.abi import PinnedBuffer
    use_dist = world > 1
    if use_dist:
        os.environ.setdefault("NCCL_DEBUG", "WARN")      # keep stdout to the one JSON line
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = local_rank if use_dist else 0
    torch.cuda.set_device(dev)
    numa_cpus = pin_to_gpu_numa(dev)        # pinned buffers are allocated (first touched) on the GPU's own NUMA node

    nb = N_SOCKETS * ((int(args.run_mib * (1 << 20)) - 112 + 15) // 16 * 16)
    buf = PinnedBuffer(nb); data = buf.array
    runs, n_full, nbytes = fill_batch_plain(data, args.run_mib, rank, world, payload=args.payload, checksum=args.checksum, kind=args.payload_kind)
    from brpc_b200 import shard
    assert np.all(shard.owner_of(runs["socket_id"], world) == rank)
    mk = lambda: brpc_b200.Context(device=dev, max_batch_bytes=nbytes + (1 << 20), max_msgs=n_full + 4096,
                                   max_runs=N_SOCKETS, tile_bytes=args.tile, max_resp_bytes=2 * nbytes + 96 * n_full + (8 << 20))
    ctx = mk()

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- correctness gate before timing: every message echoed, lengths obey the frame law -------
    rs, msgs, resp, info = ctx.process_batch_ptr(buf.ptr, nbytes, runs)
    assert len(msgs) == n_full and np.all(msgs["status"] == 0), "bench batch did not echo cleanly"
    req_bytes = int(rs["consumed"].sum())
    resp_frame_bytes = int(msgs["resp_len"].sum())
    n_msgs = len(msgs)

    # ---- value: resident batches, kernel pipeline only -----------------------------------------
    # `--pipeline D` contexts (own buffers + stream) hold the same batch; passes alternate over them so the latency-bound
    # front stages of one pass overlap the bandwidth kernel of another.  A STEP is one pass over the batch.
    depth = max(1, args.pipeline)
    ctxs = [ctx] + [mk() for _ in range(depth - 1)]
    for cx in ctxs:
        cx.upload_ptr(buf.ptr, nbytes, runs)
    for s_ in range(warmup * depth):
        ctxs[s_ % depth].launch()
    for cx in ctxs:
        cx.wait()
    launches_per_pass = ctx.execute()[1]
    fused = ctx.batch_info()["fused"]
    for cx in ctxs:
        cx.wait()
    sampler = ClockSampler(dev); sampler.start()
    barrier()
    t0 = time.perf_counter()
    for s_ in range(steps):
        ctxs[s_ % depth].launch()
    for cx in ctxs:
        cx.wait()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    dev_ms = max(ctxs[0].elapsed_ms_to(cx) for cx in ctxs[:min(depth, steps)])
    n_launch = steps * launches_per_pass
    for cx in ctxs[1:]:       # every in-flight copy produced the same, correct result
        r2, m2, p2, _ = cx.download()
        assert len(m2) == n_full and np.array_equal(m2["resp_len"], msgs["resp_len"]) and np.array_equal(m2["status"], msgs["status"])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *ctxs[(steps - 1) % depth].download()[:3])
    # per-stage device times (CUDA events between the launches of one pass), averaged
    stage_acc = {}
    for _ in range(5):
        ctx.execute()
        for name, ms in ctx.stage_times():
            stage_acc.setdefault(name, []).append(ms)
    stages = {k: statistics.mean(v) for k, v in stage_acc.items()}

    # ---- e2e: host buffers, copies inside the timed region --------------------------------------
    # Three contexts in flight (submit/collect halves of b2_process_batch): the transfers of one batch overlap the kernels of
    # the next.  Three ways of crossing PCIe, all bit-exact (tests/test_gpu_modes.py):
    #   copy      H2D copy of every request byte, D2H copy of descriptors + every reply byte (round 1's e2e)
    #   by_ref    H2D copy; replies come back as {<= 64-byte prefix, reference into the request bytes} (SendRpcResponse's own
    #             append-by-reference): D2H = descriptors + refs + prefixes
    #   pull      no H2D copy: the kernels read the pinned request blocks in place, one 128-byte row per message + the scan
    #             windows cross the link; replies by reference.  THE HEADLINE: what a brpc GpuTransport would run.
    e2e_depth = 3
    while len(ctxs) < e2e_depth:
        ctxs.append(mk())

    def e2e_mode(im, rm, min_s):
        for cx in ctxs[:e2e_depth]:
            cx.set_modes(im, rm)
            cx.process_batch_ptr(buf.ptr, nbytes, runs); cx.process_batch_ptr(buf.ptr, nbytes, runs)
        info_ = ctxs[0].batch_info()
        t1 = time.perf_counter()
        r3, m3, p3, i3 = ctxs[0].process_batch_ptr(buf.ptr, nbytes, runs)
        one = time.perf_counter() - t1
        n_steps = max(9, int(np.ceil(min_s / max(one / 2, 1e-6))))
        if use_dist:
            t_n = torch.tensor([n_steps], dtype=torch.int64, device="cuda"); dist.all_reduce(t_n, op=dist.ReduceOp.MAX); n_steps = int(t_n.item())
        barrier()
        t1 = time.perf_counter()
        for s_ in range(min(e2e_depth, n_steps)):
            ctxs[s_].submit_ptr(buf.ptr, nbytes, runs)
        ok = True
        for s_ in range(n_steps):
            cx = ctxs[s_ % e2e_depth]
            r3, m3, p3, i3 = cx.collect()
            ok = ok and len(m3) == n_full and int(m3["resp_len"][-1]) == int(msgs["resp_len"][-1])
            if s_ + e2e_depth < n_steps:
                cx.submit_ptr(buf.ptr, nbytes, runs)
        barrier()
        ms = (time.perf_counter() - t1) * 1e3 / n_steps
        assert ok, "e2e batches returned wrong results"
        if rm == 1:
            refs = i3["refs"]
            assert refs is not None and np.all(refs["src_len"] + refs["prefix_len"] == m3["resp_len"])
        if rm == 2:
            iov = i3["iov"]
            assert iov is not None and np.all(iov["len"][0::2] + iov["len"][1::2] == m3["resp_len"]) and int(r3["n_unanswered"].sum()) == 0
        d2h = int(len(m3) * 64 + len(r3) * 32 + int(r3["resp_bytes"].sum()) + (16 * rm * len(m3) if rm else 0))
        meta = int(runs.nbytes + 4 * (len(runs) + 1) + 16 * info_["n_tiles"])
        # pull: each message's stashed row is one 96-byte (by-ref; else 128-byte) PCIe read; every tile's speculative entry scan reads two 512-byte windows
        h2d = meta + (int((96 if rm else 128) * len(m3) + 1024 * info_["n_tiles"]) if im else int(nbytes))
        return {"ms_per_step": ms, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": n_steps, "tile_bytes": info_["tile_bytes"]}

    #   iovec     pull, and the device also writes the writev gather list of the replies (what b2::GpuTransport runs: e2e_messenger)
    e2e_modes = {"copy": e2e_mode(0, 0, 0.4), "copy_by_ref": e2e_mode(0, 1, 0.4), "pull_by_ref": e2e_mode(1, 1, 0.6), "pull_iovec": e2e_mode(1, 2, 0.4)}
    clocks = sampler.stop()
    for cx in ctxs:
        cx.set_modes(0, 0)

    # ---- latency: one small batch at a time (p99 of the metric) -----------------------------------
    # 64 connections x 1 complete 1 KB request each = what 64 synchronous client threads (multi_threaded_echo_c++
    # -thread_num=64) have in flight; pinned host buffers; timed inside the library (b2_latency_probe) around
    #   ring:     b2_ring_submit + b2_ring_wait — the persistent kernel, no launch / memcpy / sync per batch
    #   blocking: b2_process_batch — one k_small launch + two copies + a stream sync
    latency = None
    if not args.no_latency:
        lib, Spec = load_press()
        lib.b2press_frame.restype = C.c_size_t
        lib.b2press_frame.argtypes = [C.POINTER(Spec), C.c_uint64, C.c_void_p, C.c_size_t]
        sp = Spec(b"example.EchoService", b"Echo", PAYLOAD, 0, 0, 0, 20260921)
        tmp = C.create_string_buffer(4096)
        flen = lib.b2press_frame(C.byref(sp), 12345, tmp, 4096)
        stride = (flen + 15) // 16 * 16
        lbuf = PinnedBuffer(N_SOCKETS * stride)
        lruns = np.zeros(N_SOCKETS, dtype=RUN_DT)
        for s_ in range(N_SOCKETS):
            n_ = lib.b2press_frame(C.byref(sp), (s_ << 32) + 7, lbuf.ptr + s_ * stride, stride)
            lruns[s_] = (s_, s_ * stride, n_, 1, 0)
        lat_ctx = brpc_b200.Context(device=dev, max_batch_bytes=1 << 20, max_msgs=4096, max_runs=N_SOCKETS, tile_bytes=args.tile)
        lrs, lm, lresp, _i = lat_ctx.process_batch_ptr(lbuf.ptr, N_SOCKETS * stride, lruns)
        assert len(lm) == N_SOCKETS and np.all(lm["status"] == 0)
        lat_ctx.latency_probe(lbuf.ptr, N_SOCKETS * stride, lruns, 200, False)
        blk = np.sort(lat_ctx.latency_probe(lbuf.ptr, N_SOCKETS * stride, lruns, 3000, False))
        pc = lambda v, q: float(v[min(len(v) - 1, int(len(v) * q))])
        ring = {}
        for label, rm in (("by_ref", 1), ("copy", 0)):
            lat_ctx.set_modes(0, rm)
            lat_ctx.ring_start()
            lat_ctx.latency_probe(lbuf.ptr, N_SOCKETS * stride, lruns, 200, True)
            r0 = lat_ctx.ring_launches()
            us = np.sort(lat_ctx.latency_probe(lbuf.ptr, N_SOCKETS * stride, lruns, 5000, True))
            launches = lat_ctx.ring_launches() - r0
            t_ = lat_ctx.ring_submit(None, lruns, ptr=lbuf.ptr, nbytes=N_SOCKETS * stride)
            qrs, qm, qresp, qi = lat_ctx.ring_wait(t_)
            assert len(qm) == N_SOCKETS and np.all(qm["status"] == 0) and np.array_equal(qm["resp_len"], lm["resp_len"])
            if rm:
                assert qi["refs"] is not None and np.all(qi["refs"]["src_len"] == PAYLOAD)
            ring[label] = {"p50_us": pc(us, .5), "p99_us": pc(us, .99), "mean_us": float(us.mean()), "iters": len(us), "kernel_launches_per_batch": launches / float(len(us)),
                           "device_phase_ns": dict(zip(["header_read", "bytes_pulled", "body_done", "results_pushed"], lat_ctx.ring_phase_ns(t_)))}
            lat_ctx.ring_stop()
        lat_ctx.set_modes(0, 0)
        latency = {"batch": "%d connections x 1 request (1 KB), pinned host buffers, timed inside the library" % N_SOCKETS,
                   "path": "persistent kernel + submit ring (b2_ring_submit / b2_ring_wait)", "mode": "replies by reference (B2_RESP_BY_REF)",
                   "p50_us": ring["by_ref"]["p50_us"], "p99_us": ring["by_ref"]["p99_us"], "mean_us": ring["by_ref"]["mean_us"], "iters": ring["by_ref"]["iters"],
                   "kernel_launches_per_batch": ring["by_ref"]["kernel_launches_per_batch"], "device_phase_ns": ring["by_ref"]["device_phase_ns"],
                   "ring_copy_replies": ring["copy"],
                   "blocking_call": {"p50_us": pc(blk, .5), "p99_us": pc(blk, .99), "kernel_launches_per_batch": int(_i["n_launches"]), "iters": len(blk)}}

    # ---- reduce over ranks: max time, summed messages; NCCL all-reduce of the bvar-like counters --
    tv = [dev_ms, wall_ms] + [e2e_modes[k]["ms_per_step"] for k in ("copy", "copy_by_ref", "pull_by_ref", "pull_iovec")]
    t_dev = torch.tensor(tv, dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(n_full)], dtype=torch.float64, device="cuda")
    if use_dist:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        counters = torch.tensor(ctx.counters(), dtype=torch.int64, device="cuda")
        dist.all_reduce(counters, op=dist.ReduceOp.SUM)      # Adder semantics (bvar/reducer.h:335)
        counters = counters.tolist()
    else:
        counters = ctx.counters()
    dev_ms_max, wall_ms_max, e_copy, e_ref, e_pull, e_iov = t_dev.tolist()
    total_msgs = tot.item()
    ms_per_step = dev_ms_max / steps
    value = total_msgs / (ms_per_step * 1e-3)

    if rank == 0:
        config["value_path"] = "k_fused (decode + echo + pack in one pass)" if fused else "slot-scan pipeline (k_decode, k_scan_blocks, k_pack_tma)"
        # roofline of the dominant kernel, from THIS rank's stage times
        dom = max(stages, key=stages.get)
        pipe_alg = float(req_bytes + resp_frame_bytes + DESC_BYTES * n_msgs)                  # SURVEY §8d: req + resp + 64 B desc
        pack_alg = float(resp_frame_bytes + n_msgs * (args.payload + DESC_BYTES))             # k_pack_tma: resp written + payload & desc read
        dom_alg = {"pack": pack_alg, "fused": pipe_alg}.get(dom, pipe_alg)
        achieved = dom_alg / (stages[dom] * 1e-3) / 1e9
        pipe_ms = sum(stages.values())                                                            # one pass alone (serial stages)
        step_ms_rank0 = dev_ms / steps                                                            # with `depth` passes in flight
        mk_e2e = lambda ms_, m_: {"value": total_msgs / (ms_ * 1e-3), "unit": "msgs/s", "h2d_bytes_per_step": m_["h2d_bytes_per_step"],
                                  "d2h_bytes_per_step": m_["d2h_bytes_per_step"], "ms_per_step": ms_, "steps": m_["steps"]}
        e2e = mk_e2e(e_pull, e2e_modes["pull_by_ref"])
        e2e["mode"] = "pull_by_ref"
        e2e["note"] = ("b2_batch_submit/collect (the two halves of b2_process_batch) on pinned host blocks, 3 batches in flight, B2_INPUT_PULL + "
                       "B2_RESP_BY_REF: the kernels read the pinned request blocks in place (h2d = one 96-byte row per message + the scan windows "
                       "+ run/tile records, counted from the access pattern), replies come back as prefix + reference; e2e_modes holds the copy variants")
        line = {"metric": "echo QPS, 1 KB baidu_std", "value": value, "unit": "msgs/s", "n_gpus": world if use_dist else 1,
                "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
                "e2e": e2e,
                "e2e_modes": {"copy": mk_e2e(e_copy, e2e_modes["copy"]), "copy_by_ref": mk_e2e(e_ref, e2e_modes["copy_by_ref"]), "pull_by_ref": mk_e2e(e_pull, e2e_modes["pull_by_ref"]),
                              "pull_iovec": mk_e2e(e_iov, e2e_modes["pull_iovec"])},
                "gpu_launches": int(n_launch),
                "roofline": {"bound": "hbm", "kernel": "k_" + dom, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                             "frac": achieved / hbm_peak, "traffic": ncu_traffic("k_" + dom, args), "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": dom_alg, "kernel_ms": stages[dom]},
                "roofline_pipeline": {"achieved": pipe_alg / (step_ms_rank0 * 1e-3) / 1e9,
                                      "frac": pipe_alg / (step_ms_rank0 * 1e-3) / 1e9 / hbm_peak,
                                      "algorithmic_bytes_per_msg": pipe_alg / n_msgs, "single_pass_ms": pipe_ms, "launches_per_pass": int(launches_per_pass),
                                      "stage_ms": stages, "note": "whole hot path: (req + resp + 64 B desc) x msgs / measured time per pass"},
                "latency": latency, "clocks": clocks, "wall_ms_per_step": wall_ms_max / steps,
                "value_by_wall_clock": total_msgs * steps / (wall_ms_max * 1e-3), "msgs_per_step": total_msgs,
                "counters_allreduced": counters}
        if not use_dist and N_SOCKETS == 64 and args.run_mib >= 1:      # (the C++ bench has 64 connections of whole MiB)
            # the same e2e through the C++ host side a brpc transport would run (b2::GpuTransport: registered read regions, 8 groups of
            # connections = 8 batches in flight driven by 4 host threads, B2_INPUT_PULL + B2_RESP_IOVEC: the device writes the gather list
            # and every connection's replies leave through writev (into /dev/null) as they stand; tests/cpp/transport_test.cc bench)
            tb = os.path.join(ROOT, "tests", "cpp", "transport_test")
            if os.path.exists(tb):
                try:
                    for cx in ctxs:
                        cx.close()
                    out = subprocess.run([tb, "bench", str(int(args.run_mib)), "40", "1", "2", "8", "2"], capture_output=True, text=True, timeout=120)
                    line["e2e_messenger"] = json.loads(out.stdout.strip().splitlines()[-1]) if out.returncode == 0 else {"error": (out.stderr or out.stdout)[-300:]}
                except Exception as e:      # noqa: BLE001
                    line["e2e_messenger"] = {"error": repr(e)}
        if not args.no_cpu_baseline and not use_dist:
            # (rank 0 at N = 1 only) bounded sample: the first 8 connections of the same batch, 1 thread, ~10 s
            sub = runs[:8].copy()
            q1, m1, p1 = cpu_arm(data, sub, 1, min_seconds=8.0)
            line["cpu_baseline"] = {"value": q1, "unit": "msgs/s", "cores": 1, "kind": "port",
                                    "sample": "8 of the %d connections (%d msgs/pass), best of %d passes, single thread" % (N_SOCKETS, m1, p1)}
        print(json.dumps(line))
    if use_dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
