"""GPU: `bench.py --dump-outputs DIR` — the same arguments write the same float32 / float64 files, within 64 MB, and what they
hold for the timed batch is what the oracle computes for it, but for where the replies sit in the reply buffer."""
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest

import _oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def test_dump_outputs_repeat_and_match_the_oracle(tmp_path):
    args = ("--steps", "3", "--warmup", "3", "--run-mib", "0.25", "--no-cpu-baseline", "--no-latency")
    for d in ("a", "b"):
        p = subprocess.run([sys.executable, BENCH, *args, "--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and "reply_bytes.npy" in names
    out, total = {}, 0
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), n
        out[n[:-4]] = a
        total += os.path.getsize(tmp_path / "a" / n)
    assert total <= 64 << 20

    spec = importlib.util.spec_from_file_location("bench", BENCH)
    bench = importlib.util.module_from_spec(spec); spec.loader.exec_module(bench)
    data = np.zeros(bench.N_SOCKETS * ((int(0.25 * (1 << 20)) - 112 + 15) // 16 * 16), np.uint8)
    runs, n_full, nbytes = bench.fill_batch_plain(data, 0.25, 0, 1)
    rs, msgs, resp = O.process_batch(O.make_config(), data, runs, resp_cap=2 * nbytes + 96 * n_full + (8 << 20))
    bench.dump_outputs(str(tmp_path / "oracle"), rs, msgs, resp)
    layout = {"msg_resp_off", "run_resp_off", "run_resp_bytes", "run_msgs_crc32"}    # where replies sit in the buffer is the device's choice
    assert len(out["msg_index"]) == min(4096, n_full) and "run_reply_crc32" in out
    for k, a in out.items():
        if k not in layout:
            assert np.array_equal(a, np.load(tmp_path / "oracle" / (k + ".npy"))), k
