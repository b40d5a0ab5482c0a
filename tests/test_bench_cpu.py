"""CPU check of bench.py's reference arm (the unmodified reference timed on the host cores) and of the
JSON contract keys; uses BASELINE config 1 (256x256, 4 spp) so it runs in seconds."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT
from oracle import ref


@pytest.mark.skipif(not ref.available(), reason="oracle/_ref not built")
def test_reference_arm_json_contract():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1",
                        "--steps", "1", "--warmup", "0", "--sqrtspp", "2"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "Mray/s" and line["value"] > 0
    assert line["vs_baseline"] is None and line["higher_is_better"] is True
    assert set(line["cpu_baseline"]) >= {"value", "unit", "cores", "kind", "sample"} and line["cpu_baseline"]["kind"] == "reference"
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"]


def load_bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_dump_outputs_writer(tmp_path, monkeypatch):
    """bench.py --dump-outputs: the frame as image.npy; over the size limit, the same seeded pixel sample every time."""
    import numpy as np
    bench = load_bench()
    frame = np.random.default_rng(1).random((6, 8, 3), dtype=np.float32)
    bench.write_outputs(str(tmp_path / "full"), frame)
    assert np.array_equal(np.load(tmp_path / "full" / "image.npy"), frame)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 400)
    for run in ("a", "b"):
        bench.write_outputs(str(tmp_path / run), frame)
    a = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in ("image_sample", "image_sample_index")}
    assert sum(v.nbytes for v in a.values()) <= 400 and a["image_sample_index"].dtype == np.float64
    assert np.array_equal(a["image_sample"], frame.reshape(-1, 3)[a["image_sample_index"].astype(int)])
    for n, v in a.items():
        assert np.array_equal(np.load(tmp_path / "b" / (n + ".npy")), v)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.main()


def test_ncu_epilogue_parser():
    """bench.py's non-timed ncu epilogue: per-kernel DRAM bytes / FP64 instructions / lanes from `ncu --csv` rows and the
    child's counters (a synthetic capture; the real one runs on the GPU box)."""
    bench = load_bench()
    hdr = '"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size","Device","CC","Section Name","Metric Name","Metric Unit","Metric Value"'

    def row(i, kernel, metric, unit, value):
        return f'"{i}","1","python","h","{kernel}","1","13","(256, 1, 1)","(2368, 1, 1)","0","10.0","Command line profiler metrics","{metric}","{unit}","{value}"'
    lines = ["==PROF== Connected", hdr]
    for i, (kernel, rd, wr) in enumerate([("void mcrt::k_extend<double, 1, 1>(mcrt::WaveParams<T1>, int)", "1,000", "200"),
                                          ("void mcrt::k_extend<double, 1, 1>(mcrt::WaveParams<T1>, int)", "3000", "800"),
                                          ("void mcrt::k_shade_key<double>(mcrt::WaveParams<T1>)", "5", "5"),
                                          ("void mcrt::k_shade<double, 0, 0, 4294967282>(mcrt::WaveParams<T1>, int)", "2", "2")]):
        lines += [row(i, kernel, "gpu__time_duration.sum", "ns", "1000"), row(i, kernel, "dram__bytes_read.sum", "byte", rd),
                  row(i, kernel, "dram__bytes_write.sum", "Kbyte" if i == 3 else "byte", wr),
                  row(i, kernel, "smsp__sass_thread_inst_executed_op_dfma_pred_on.sum", "inst", "100"),
                  row(i, kernel, "smsp__sass_thread_inst_executed_op_dmul_pred_on.sum", "inst", "50"),
                  row(i, kernel, "smsp__sass_thread_inst_executed_op_dadd_pred_on.sum", "inst", "50"),
                  row(i, kernel, "smsp__thread_inst_executed.sum", "inst", "6400"), row(i, kernel, "smsp__inst_executed.sum", "inst", "400")]
    lines.append('CHILD_STATS ' + json.dumps({"extension_rays": 100, "shadow_rays": 50, "knn_queries": 0}))
    out = bench.parse_ncu_output("\n".join(lines))
    assert set(out) == {"k_extend", "k_shade"}                 # k_shade_key is not k_shade; no shadow / k-NN launches in the capture
    assert out["k_extend"]["launches"] == 2 and out["k_extend"]["dram_bytes_per_unit"] == (1000 + 200 + 3000 + 800) / 100
    assert out["k_extend"]["fp64_thread_inst_per_unit"] == 400 / 100 and out["k_extend"]["lanes_per_inst"] == 16.0
    assert out["k_shade"]["dram_bytes_per_unit"] == (2 + 2000) / 100        # Kbyte row scaled to bytes
    assert "unavailable" in bench.parse_ncu_output("no counters here")
