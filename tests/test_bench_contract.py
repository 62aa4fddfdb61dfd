"""CPU-only checks of the measurement plumbing: the CPU arm's JSON contract, the FLOP accounting bench.py divides
by, and the ncu launch-list summariser's step isolation."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--cpu-batch", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "images/sec" and d["unit"] == "images/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    # the reference's own modules when oracle/_ref is populated (build() does it when the reference is readable)
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "agedb-dir", "fds.py"))
    assert d["cpu_baseline"]["kind"] == ("reference" if have_ref else "port") and d["cpu_baseline"]["cores"] >= 1
    assert "IMDB-WIKI" in d["config"]["workload"] and "fds_ms" in d["cpu_baseline"]
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and d["gpu_launches"] == 0


def test_bench_rejects_zero_steps_and_a_dump_of_the_cpu_arm():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                           timeout=600, cwd=ROOT)
        assert r.returncode == 2 and extra[-2] in r.stderr, (extra, r.stderr[-2000:])


def test_conv_flop_accounting_matches_survey():
    sys.path.insert(0, ROOT)
    import bench
    f, d, w = bench.conv_flops_per_image()
    # SURVEY 8(d): 8.174 GFLOP forward (4.087 GMAC incl. the 2048->1 regressor, negligible), fwd+bwd = 3 x fwd - conv1 dgrad
    assert abs(f / 1e9 - 8.174) < 0.02
    assert w == f and abs((f + d + w) / 1e9 - 24.29) < 0.06
    stem = 2.0 * 112 * 112 * 64 * 3 * 49
    assert abs((f - d) - stem) < 1.0


def test_launch_list_summariser_isolates_one_step(tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import summarize
    rows = ['"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size",'
            '"Device","CC","Section Name","Metric Name","Metric Unit","Metric Value"']
    names = ["setup_kernel", "dirb200::prep_weights_all_kernel(x)", "dirb200::igemm_kernel<256, 0, 0, 0, 0, 1>(a)",
             "dirb200::bn_stats_kernel(b)", "dirb200::adam_kernel(c)", "dirb200::prep_weights_all_kernel(x)",
             "dirb200::igemm_kernel<256, 0, 0, 0, 0, 1>(a)", "dirb200::adam_kernel(c)"]
    for i, n in enumerate(names):
        for metric, unit, val in (("gpu__time_duration.sum", "us", "10"), ("dram__bytes_read.sum", "Mbyte", "100"),
                                  ("dram__bytes_write.sum", "Mbyte", "50")):
            rows.append(f'"{i}","1","python","h","{n}","1","7","(256, 1, 1)","(148, 1, 1)","0","10.0","Command line profiler metrics","{metric}","{unit}","{val}"')
    src = tmp_path / "launches.csv"
    src.write_text("==PROF== header\n" + "\n".join(rows) + "\n")
    dst = tmp_path / "out.md"
    summarize.launches(str(src), str(dst))
    summary = json.loads((tmp_path / "out.json").read_text())
    # step = (first adam, second adam]: weight prep, one conv, adam
    assert summary["conv_launches"] == 1 and abs(summary["conv_ms"] - 0.01) < 1e-9
    assert abs(summary["conv_dram_gb"] - 0.15) < 1e-9
    assert "ONE training step (3 launches" in dst.read_text()
