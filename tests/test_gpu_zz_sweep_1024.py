"""GPU parity at BASELINE configs[2]'s SHAPE (SURVEY §8(d), config 3): 1024 sockets in ONE batch, every payload size of the rpc_press sweep
(64 B ... 64 KiB, 11 sizes), requests drawn round-robin from a short message list like rpc_press's `_msgs`
(tools/rpc_press/rpc_press_impl.cpp:232), message bytes constant 'r' or the 62-character table of
test/brpc_snappy_compress_unittest.cpp:203, request_compress_type in {none, snappy} (rpc_press.cpp:41-42) and the request checksum on / off
(example/echo_c++/client.cpp:76-78) — the CUDA path through the C ABI against the oracle, bit for bit: run statuses, descriptors and reply bytes.
Every run ends in the middle of a frame (the socket's next read would complete it), so 1024 tails are carried per batch.
On a GPU each socket holds 256 KiB of pending bytes (the sweep's setting, profiles/r2_sweep.sh); on the emulated library (tests/emul_runner.py,
no GPU) the runs are a few frames long and two of the sizes are run (B2_SWEEP_SIZES=64,1024,... picks others), so that the file finishes in minutes — 1024 runs per batch either way."""
import os
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import _oracle as O  # noqa: E402
from _compare import assert_same  # noqa: E402
from _traffic import SEED, rnd62  # noqa: E402

N_SOCKETS = 1024
EMUL = bool(os.environ.get("B2_EMUL_LIB"))
SIZES = [64, 1024] if EMUL else [64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536]
if os.environ.get("B2_SWEEP_SIZES"):
    SIZES = [int(x) for x in os.environ["B2_SWEEP_SIZES"].split(",")]
N_MSGS = 8                                   # length of the round-robin list


def _message(rng, n, kind):
    if kind == "r":
        return b"r" * n
    if kind == "rnd":
        return rnd62(rng, n)
    return rnd62(rng, n // 2) + b"r" * (n - n // 2)           # "mix": snappy shrinks it to about a half, replies stay <= 2 x the input


def _streams(rng, n, kind, compress, checksum, run_bytes):
    frames = [O.pack_echo_request(log_id=k, correlation_id=(k + 1) << 8 | 1, message=_message(rng, n, kind), compress_type=compress,
                                  checksum_type=checksum) for k in range(N_MSGS)]
    ring = b"".join(frames)
    starts = [0]
    for f in frames:
        starts.append(starts[-1] + len(f))
    reps = run_bytes // len(ring) + 2
    long = ring * reps
    out = []
    for s in range(N_SOCKETS):
        at = starts[s % N_MSGS]                                # socket s starts at message s of the list
        cut = run_bytes - (s % 7)                              # ragged: not every run has the same length
        out.append(long[at:at + cut])
    return out, max(len(f) for f in frames)


def _run_bytes(n, compress):
    frame = n + 80
    if EMUL:
        return int(frame * 2.5) + 97
    if compress:
        return max(96 << 10, int(frame * 1.5)) + 97           # (replies are the UNcompressed messages: keep the reply arena moderate)
    return (256 << 10) - 77


@pytest.fixture(scope="module")
def ctx():
    import brpc_b200
    c = brpc_b200.Context(device=0, max_batch_bytes=(64 << 20) if EMUL else (288 << 20), max_msgs=(1 << 18) if EMUL else (1 << 22),
                          max_runs=N_SOCKETS, max_resp_bytes=(192 << 20) if EMUL else (640 << 20))
    yield c
    c.close()


CASES = [("r", 0, 0), ("rnd", 0, 1), ("mix", 1, 0), ("mix", 1, 1)]


@pytest.mark.parametrize("kind,compress,checksum", CASES, ids=["plain", "crc32c", "snappy", "snappy+crc32c"])
def test_sweep_sizes_with_1024_sockets_per_batch(ctx, kind, compress, checksum):
    import brpc_b200
    cfg = O.make_config()
    for n in SIZES:
        rng = random.Random(SEED + n + 7 * compress + 13 * checksum)
        chunks, frame_max = _streams(rng, n, kind, compress, checksum, _run_bytes(n, compress))
        data, runs = brpc_b200.make_runs(chunks)
        assert len(runs) == N_SOCKETS
        dev = ctx.process_batch(data, runs)
        orc = O.process_batch(cfg, data, runs)
        what = "payload=%d kind=%s compress=%d checksum=%d" % (n, kind, compress, checksum)
        assert_same(dev, orc, what)
        rs, msgs = dev[0], dev[1]
        # every run parsed whole frames and stopped at its cut tail (NOT_ENOUGH_DATA), nothing failed
        assert np.all(rs["parse_error"] == 2) and np.all(rs["n_msgs"] >= 1), what
        assert np.all(msgs["status"] == 0) and len(msgs) == int(rs["n_msgs"].sum()), what
        assert np.all(np.asarray([len(c) for c in chunks]) - rs["consumed"] < frame_max), what
