"""CPU tests: the oracle against the committed golden vectors (tests/golden/).

These pin the oracle (SURVEY §8c): CRC-32C to the RFC 3720 vectors the reference
asserts in test/crc32c_unittest.cc:18-71 (values re-derived through the
reference's own crc32c.cc), the protobuf wire codec to python-protobuf's
accept/reject verdicts and decoded fields, and the BASELINE 46 B / 18 B metas.
"""
import json
import os

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
G = os.path.join(HERE, "golden")

H = dict(REQUEST=1 << 0, RESPONSE=1 << 1, COMPRESS=1 << 2, CID=1 << 3, ATT=1 << 4, CHUNK=1 << 5, AUTH=1 << 6,
         SS=1 << 7, UF=1 << 8, CT=1 << 9, CKT=1 << 10, CKV=1 << 11, LOG=1 << 12, TRACE=1 << 13, RID=1 << 14, TMO=1 << 15)


def load(name):
    with open(os.path.join(G, name)) as f:
        return json.load(f)


def test_crc32c_kat(oracle):
    for k in load("crc32c_kat.json"):
        b = bytes.fromhex(k["hex"])
        if k["name"].startswith("extend"):
            assert oracle.crc32c(b[6:], oracle.crc32c(b[:6])) == k["expect"]
            continue
        assert oracle.crc32c(b) == k["crc"], k["name"]
        if "expect" in k:
            assert oracle.crc32c(b) == k["expect"]
        if "masked" in k:
            assert oracle.lib.orc_crc32c_mask(k["crc"]) == k["masked"]
            assert oracle.lib.orc_crc32c_unmask(k["masked"]) == k["crc"]


def test_snappy_matches_the_reference_results(oracle):
    """The oracle's snappy against the vendored snappy 1.1.3: compressed bytes of snappy_vectors.json, RawUncompress's
    verdict and output on the corrupted streams of snappy_ref_results.json."""
    import random
    import _snappy_cases as S
    from _traffic import SEED
    seeds = []
    for v in load("snappy_vectors.json"):
        raw = bytes.fromhex(v["raw_hex"]) if "raw_hex" in v else (b"abcdefghijklmnopqrstuvwxyz0123456789" * (v["raw_len"] // 36 + 1))[:v["raw_len"]]
        comp = bytes.fromhex(v["comp_hex"])
        assert oracle.snappy_compress(raw) == comp, v["name"]
        assert oracle.snappy_uncompressed_length(comp) == len(raw) and oracle.snappy_uncompress(comp, len(raw)) == raw, v["name"]
        if 0 < len(comp) < 5000:
            seeds.append(comp)
    want = S.ref_results()["gpu_corruptions"]
    blobs = S.corrupted_blobs(random.Random(SEED), seeds)
    assert len(blobs) == len(want)
    for b, w in zip(blobs, want):
        ul = oracle.snappy_uncompressed_length(b)
        got = oracle.snappy_uncompress(b, ul) if ul is not None and ul <= 32 * len(b) + 64 else None
        assert S.digest(got) == w, b.hex()[:80]


def span(b, s):
    return b[s.off:s.off + s.len].hex()


def check_meta(b, m, f):
    has = m.has
    assert bool(has & H["REQUEST"]) == f["has_request"]
    if f["has_request"]:
        assert span(b, m.service_name) == f["service_name"]
        assert span(b, m.method_name) == f["method_name"]
        assert bool(has & H["LOG"]) == f["has_log_id"] and m.log_id == f["log_id"]
        assert bool(has & H["TRACE"]) == f["has_trace_id"] and m.trace_id == f["trace_id"]
        assert bool(m.has_span_id) == f["has_span_id"] and m.span_id == f["span_id"]
        assert bool(m.has_parent_span_id) == f["has_parent_span_id"] and m.parent_span_id == f["parent_span_id"]
        assert bool(has & H["TMO"]) == f["has_timeout_ms"] and m.timeout_ms == f["timeout_ms"]
        assert bool(has & H["RID"]) == f["has_request_id"]
        if f["has_request_id"]:
            assert span(b, m.request_id) == f["request_id"]
    assert bool(has & H["RESPONSE"]) == f["has_response"]
    if f["has_response"]:
        assert bool(m.has_error_code) == f["has_error_code"] and m.error_code == f["error_code"]
        assert bool(m.has_error_text) == f["has_error_text"]
        if f["has_error_text"]:
            assert span(b, m.error_text) == f["error_text"]
    for bit, k in (("COMPRESS", "compress_type"), ("CID", "correlation_id"), ("ATT", "attachment_size"),
                   ("CT", "content_type"), ("CKT", "checksum_type")):
        assert bool(has & H[bit]) == f["has_" + k], k
        assert getattr(m, k) == f[k], k
    assert bool(has & H["CKV"]) == f["has_checksum_value"]
    if f["has_checksum_value"]:
        assert span(b, m.checksum_value) == f["checksum_value"]
    assert bool(has & H["AUTH"]) == f["has_authentication_data"]
    if f["has_authentication_data"]:
        assert span(b, m.authentication_data) == f["authentication_data"]
    assert bool(has & H["CHUNK"]) == f["has_chunk_info"]
    assert bool(has & H["SS"]) == f["has_stream_settings"]
    if f["has_stream_settings"]:
        assert m.ss_stream_id == f["ss_stream_id"]
        assert bool(m.ss_need_feedback) == f["ss_need_feedback"] and bool(m.ss_writable) == f["ss_writable"]
        assert m.ss_n_extra == f["ss_n_extra"]
    # upb moves a map entry that carries unknown fields to the parent's unknown set,
    # C++ MapEntry parsing keeps it; only the implication upb-sees-entries => we-do is pinned
    if f["n_user_fields_distinct"] > 0:
        assert m.n_user_fields > 0


def check_stream(m, f):
    assert bool(m.has & 1) == f["has_stream_id"] and m.stream_id == f["stream_id"]
    assert bool(m.has & 2) == f["has_source_stream_id"] and m.source_stream_id == f["source_stream_id"]
    assert bool(m.has & 4) == f["has_frame_type"] and m.frame_type == f["frame_type"]
    assert bool(m.has & 8) == f["has_has_continuation"]
    assert bool(m.has & 0x100) == bool(f["has_continuation"])
    assert bool(m.has & 16) == f["has_feedback"]
    assert bool(m.feedback_has_consumed_size) == f["feedback_has_consumed_size"]
    assert m.consumed_size == f["consumed_size"]


def test_baseline_meta_sizes():
    v = load("rpc_meta_vectors.json")["rpc_meta"]
    assert len(v[0]["hex"]) // 2 == 46 and len(v[1]["hex"]) // 2 == 18     # SURVEY §8 preamble


def test_rpc_meta_valid_vectors(oracle):
    for rec in load("rpc_meta_vectors.json")["rpc_meta"]:
        b = bytes.fromhex(rec["hex"])
        ok, m = oracle.parse_rpc_meta(b)
        assert ok, rec["note"]
        check_meta(b, m, rec["fields"])


def test_stream_meta_valid_vectors(oracle):
    for rec in load("rpc_meta_vectors.json")["stream_frame_meta"]:
        ok, m = oracle.parse_stream_meta(bytes.fromhex(rec["hex"]))
        assert ok
        check_stream(m, rec["fields"])


def test_echo_request_vectors(oracle):
    for rec in load("rpc_meta_vectors.json")["echo_request"]:
        b = bytes.fromhex(rec["hex"])
        ok, (off, ln) = oracle.parse_echo_request(b)
        assert ok == rec["ok"], rec["hex"][:80]
        if ok and "message_len" in rec:
            assert ln == rec["message_len"] and b[off:off + ln] == b"r" * ln
        if ok and "message_hex" in rec:
            assert b[off:off + ln].hex() == rec["message_hex"]


def test_pb_fuzz_vectors(oracle):
    fz = load("pb_fuzz_vectors.json")
    bad = []
    for i, rec in enumerate(fz["rpc_meta"]):
        b = bytes.fromhex(rec["hex"])
        ok, m = oracle.parse_rpc_meta(b)
        if ok != rec["ok"]:
            bad.append((i, rec["hex"], rec["ok"], ok))
            continue
        if ok:
            check_meta(b, m, rec["fields"])
    assert not bad, "verdict mismatches (idx, hex, upb, oracle): %r" % bad[:10]
    bad = []
    for i, rec in enumerate(fz["stream_frame_meta"]):
        ok, m = oracle.parse_stream_meta(bytes.fromhex(rec["hex"]))
        if ok != rec["ok"]:
            bad.append((i, rec["hex"], rec["ok"], ok))
            continue
        if ok:
            check_stream(m, rec["fields"])
    assert not bad, bad[:10]


def test_meta_fast_path_agrees_with_generic_on_golden_vectors():
    """decode_rpc_meta_fast (product, csrc/b2_core.cuh) is a host+device function: compiled here for the host,
    it must either decline or agree with the generic decoder on every golden / fuzz vector."""
    import subprocess, tempfile, struct
    root = os.path.dirname(HERE)
    src = r'''
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "brpc_b200/csrc/b2_core.cuh"
int main(int argc, char** argv) {
    FILE* f = fopen(argv[1], "rb"); unsigned n_fast = 0, n_tot = 0, bad = 0;
    for (;;) {
        unsigned len; if (fread(&len, 4, 1, f) != 1) break;
        unsigned char* b = (unsigned char*)malloc(len + 1); if (len && fread(b, 1, len, f) != len) return 2;
        b2::RpcMetaOut a, g; memset(&a, 0, sizeof a); memset(&g, 0, sizeof g);
        const bool fa = b2::decode_rpc_meta_fast(b, len, a), ge = b2::decode_rpc_meta(b, len, g);
        n_tot++;
        if (fa) { n_fast++; if (!ge || memcmp(&a, &g, sizeof a) != 0) { bad++; fprintf(stderr, "mismatch at vector %u\n", n_tot - 1); } }
        free(b);
    }
    printf("%u %u %u\n", n_tot, n_fast, bad);
    return bad ? 1 : 0;
}'''
    blobs = [bytes.fromhex(r["hex"]) for r in load("rpc_meta_vectors.json")["rpc_meta"]] + [bytes.fromhex(r["hex"]) for r in load("pb_fuzz_vectors.json")["rpc_meta"]]
    with tempfile.TemporaryDirectory() as td:
        open(os.path.join(td, "t.cc"), "w").write(src)
        with open(os.path.join(td, "v.bin"), "wb") as f:
            for b in blobs:
                f.write(struct.pack("<I", len(b))); f.write(b)
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-I", root, "-o", os.path.join(td, "t"), os.path.join(td, "t.cc")])
        out = subprocess.run([os.path.join(td, "t"), os.path.join(td, "v.bin")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    tot, fast, bad = map(int, out.stdout.split())
    assert tot == len(blobs) and bad == 0 and fast > 50
