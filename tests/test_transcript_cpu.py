"""The transcript kernels of csrc/transcript.cuh (k_text_extract -> k_text_scan -> k_text_pack) on the CPU box: compiled with
g++ over the SIMT emulator (tests/support/host_relay2.cpp) and driven through the same bodies as tests/test_transcript_gpu.py,
plus the host half (TranscriptBook / TranscriptLog) against the unmodified reference's write_log.  Test aid only."""
import os
import sys
from datetime import datetime
from pathlib import Path

import pytest

import test_transcript_gpu as G
from host_relay import HostBulkEngine
from llmapigateway_b200.transcripts import TranscriptLog, render_log


@pytest.fixture(scope="module")
def engine():
    e = HostBulkEngine(max_streams=1024, carry_cap=8192, n_blocks=2)
    e.enable_transcripts()
    yield e
    e.close_engine()


@pytest.mark.parametrize("stepping", ["one_step", "step_per_chunk", "random_steps"])
def test_golden_transcripts(engine, stepping):
    G.test_golden_transcripts(engine, stepping)


@pytest.mark.parametrize("stepping", ["one_step", "random_steps"])
def test_adversarial_content(engine, stepping):
    G.test_adversarial_content_vs_oracle(engine, stepping, n_streams=600)


@pytest.mark.parametrize("events_per_chunk", [1, 8])
def test_c3_shape(engine, events_per_chunk):
    G.test_c3_shape_takes_the_lane_parallel_path(engine, events_per_chunk, n_streams=24)


def test_mid_event_cuts(engine):
    G.test_mid_event_cuts_across_steps(engine)


def test_runs_once(engine):
    G.test_transcript_pass_runs_once_per_step(engine)


# ---- host half: write_log ---------------------------------------------------------------------------------------------------
USAGE = {"prompt_tokens": 10, "completion_tokens": 5, "total_tokens": 17, "reasoning_tokens": 2, "cached_tokens": 4, "cost": 0.00123,
         "model": "m-ok", "provider": "P"}
GOLDEN_LOG = Path(__file__).parent / "golden" / "write_log_cases.json"


def test_write_log_file_equals_the_reference_fixture(tmp_path):
    """Files written by the UNMODIFIED write_log (tests/golden/make_write_log_golden.py) vs TranscriptLog, byte for byte."""
    import json
    cases = json.loads(GOLDEN_LOG.read_text())["cases"]
    assert len(cases) >= 6
    for k, c in enumerate(cases):
        rows = []
        d = tmp_path / f"logs{k}"
        log = TranscriptLog(log_dir=str(d), usage_sink=rows.append, clock=lambda: datetime(2026, 1, 2, 3, 4, 5, 678901))
        text = c["accum"].encode("utf-8", "surrogatepass")
        log.write_log(c["headers"], c["body"], text, c["usage"])
        files = sorted(d.glob("*.txt")) if d.exists() else []
        if c["file"] is None:                                    # the reference's f.write raised: no row either
            assert rows == [] and log.failed == 1, c["name"]
            assert not files or files[0].read_bytes() != b"never", c["name"]
            continue
        assert [f.name for f in files] == ["2026-01-02_03-04-05.678.txt"], c["name"]
        assert files[0].read_bytes().decode("utf-8") == c["file"], c["name"]
        assert rows == [c["usage"]], c["name"]


def test_write_log_prunes_like_the_reference(tmp_path):
    d = tmp_path / "logs"
    t = [0]

    def clock():
        t[0] += 1
        return datetime(2026, 1, 2, 3, 4, t[0] % 60, t[0] * 1000)
    log = TranscriptLog(log_dir=str(d), log_file_limit=3, clock=clock)
    for k in range(6):
        log.write_log({}, "{}", f"text {k}", dict(USAGE))
        os.utime(sorted(d.glob("*.txt"))[-1], (1000 + k, 1000 + k))
    names = sorted(p.name for p in d.glob("*.txt"))
    assert len(names) == 3 and log.written == 6
    assert "text 5" in (d / names[-1]).read_text()


def test_render_log_blocks():
    s = render_log({"a": 1}, '{"x":"y\\n"}', "hello", USAGE)
    assert s.startswith("-" * 100 + "\nTokens Usage:\n-" + "-" * 100 + "\n\nInput: 10\nOutput: 5\nCached: 4\nReasoning: 2\nTotal: 17\nCost: $0.001230\nModel: m-ok\nProvider: P\n\n")
    assert s.endswith("LLM Response:\n" + "-" * 100 + "\n\nhello")


# ---- the seam: make_llm_request + StreamBatcher with a TranscriptLog (emulated kernels as the engine) ---------------------------
def test_gateway_writes_the_log_files_the_reference_writes(tmp_path):
    """Every golden stream through make_llm_request with transcripts on: the files written (one per write_log call, in call
    order) hold the reference's transcripts, and a usage row follows each file -- none when the write fails."""
    import asyncio
    import json
    import httpx
    from golden_io import canon_rows
    from llmapigateway_b200.gateway import StreamBatcher, make_llm_request

    def client_factory(chunks, status):
        class _Body(httpx.AsyncByteStream):
            async def __aiter__(self):
                for c in chunks:
                    yield c
        return lambda **kw: httpx.AsyncClient(transport=httpx.MockTransport(
            lambda request: httpx.Response(status, headers={"content-type": "text/event-stream"}, stream=_Body())), **kw)

    calls = []

    class Log(TranscriptLog):
        def write_log(self, h, b, text, usage):
            calls.append((h, b, bytes(text), dict(usage)))
            super().write_log(h, b, text, usage)

    async def go():
        eng = HostBulkEngine(max_streams=16, carry_cap=8192, n_blocks=1)
        rows = []
        tick = [0]

        def clock():
            tick[0] += 1
            return datetime(2026, 1, 2, 3, tick[0] // 60 % 60, tick[0] % 60, (tick[0] * 1000) % 1000000)
        log = Log(log_dir=str(tmp_path / "logs"), log_file_limit=10000, usage_sink=rows.append, clock=clock)
        batcher = StreamBatcher(eng, window_s=0.0005, transcript_log=log)
        n_cmp = 0
        for case in G.CASES[:150]:
            n0, r0 = len(calls), len(rows)
            resp, err = await make_llm_request("http://u.test/v1/chat/completions", {}, {"model": "m"}, True, batcher=batcher,
                                               client_factory=client_factory(case["chunks"], case["http_status"]),
                                               log_request=dict(req_headers={"x": case["name"]}, req_body_str='{"model":"m"}'))
            if resp is None:
                assert case["failed"] and len(calls) == n0
                continue
            _ = [c async for c in resp.body_iterator]
            got = calls[n0:]
            want_rows = json.loads(case["rows"])
            if any(h != {"x": case["name"]} or b != '{"model":"m"}' for h, b, _, _ in got):
                raise AssertionError(case["name"])
            try:
                texts = [t.decode("utf-8", "surrogatepass") for _, _, t, _ in got]
            except Exception:
                raise AssertionError(case["name"])
            if len(texts) != len(case["transcripts"]):
                continue                                   # exotic shapes are reported, not modelled (same rule as the row tests)
            assert texts == case["transcripts"], case["name"]
            writable = [not any(0xD800 <= ord(ch) <= 0xDFFF for ch in t) for t in texts]
            assert len(rows) - r0 == sum(writable), case["name"]
            try:
                got_rows = canon_rows(rows[r0:])
            except TypeError:
                continue                                   # a value the device reports as unrepresentable (big int ...): not compared
            assert got_rows == canon_rows([r for r, ok in zip(want_rows, writable) if ok]), case["name"]
            n_cmp += 1
        assert n_cmp >= 90
        return log
    log = asyncio.run(go())
    assert log.written >= 90 and len(list((tmp_path / "logs").glob("*.txt"))) == log.written
