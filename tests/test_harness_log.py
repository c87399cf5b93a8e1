"""The reference's own log parser (utils/benchmark/benchmark_results.py of vk_gltf_renderer) reads a log b200pt_headless wrote on
a B200 for the reference harness's command line (tests/golden/headless_box_harness.log, captured by
tests/test_gpu_scenes.py::test_headless_accepts_the_reference_harness_command_line).  What that parser returned for the log
(parse_headless_summary and iter_benchmark_records) is stored beside it in tests/golden/headless_box_harness_parsed.json, so
the test needs no copy of the reference tree."""
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOG = os.path.join(ROOT, "tests", "golden", "headless_box_harness.log")
PARSED = os.path.join(ROOT, "tests", "golden", "headless_box_harness_parsed.json")


def test_reference_parser_reads_our_headless_log():
    log = open(LOG).read()
    parsed = json.load(open(PARSED))
    # the log still holds exactly the schema-1 records the reference parser yielded from it
    records = [json.loads(l[l.find("BENCHMARK_JSON ") + len("BENCHMARK_JSON "):]) for l in log.splitlines() if "BENCHMARK_JSON " in l]
    assert [r for r in records if r.get("schema") == 1 and isinstance(r.get("type"), str)] == parsed["benchmark_records"]
    summary = parsed["headless_summary"]
    assert summary is not None
    assert summary["frames"] == "6" and summary["maxFrames"] == "6" and summary["ptSamples"] == "2"
    assert summary["effective_spp"] == "12" and summary["measured_effective_spp"] == "10"
    assert summary["warmup_frames"] == "1" and summary["measured_frames"] == "5"
    assert summary["resolution_w"] == "96" and summary["resolution_h"] == "64"
    assert float(summary["wall_ms"]) > 0 and float(summary["ms_per_frame"]) > 0 and float(summary["throughput_MSps"]) > 0
    # every summary field the parser extracted is the headless_summary record's value
    rec = [r for r in records if r["type"] == "headless_summary"][0]
    assert all(abs(float(v) - float(rec[k])) <= 5e-4 * max(1.0, abs(float(rec[k]))) for k, v in summary.items())
    records = parsed["benchmark_records"]
    assert records and records[-1]["type"] == "headless_summary" and records[-1]["backend"] == "b200pt"
