"""bench.py's JSON contract: the committed round-1 lines (measured on the B200) and a live run of the
CPU reference arm carry every key the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def _check_common(d):
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["metric"] == "mel_frames_per_sec" and d["unit"] == "mel-frames/s" and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
    assert d["value"] > 0 and d["ms_per_step"] > 0


def test_committed_engine_lines_have_the_contract_keys():
    for name, n in (("r01_bench_final_fp32.json", 1), ("r01_bench_final_tf32.json", 1), ("r01_bench_final_2gpu_fp32.json", 2)):
        d = json.load(open(os.path.join(ROOT, "profiles", name)))
        _check_common(d)
        assert d["n_gpus"] == n and d["warmup"] >= 3 and d["gpu_launches"] > 0
        assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
        assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        r = d["roofline"]
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] in ("hbm", "tensor")
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
        assert d["parity"]["durations_identical"] is True
    d = json.load(open(os.path.join(ROOT, "profiles", "r01_bench_final_fp32.json")))
    cb = d["cpu_baseline"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(cb) and cb["kind"] in ("port", "reference")
    assert d["parity"]["wav_rms_err_over_rms"] < 1e-4 and d["parity"]["mel_max_abs_err_over_max_abs"] < 1e-4


def _load_bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_reference_arm_runs_on_cpu_and_prints_one_compact_json_line(tmp_path):
    dump = tmp_path / "outputs"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--dump-outputs", str(dump)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and len(lines[0]) < 4096
    d = json.loads(lines[0])
    _check_common(d)
    assert d["impl"] == "reference" and d["steps"] == 1 and d["warmup"] == 1 and d["gpu_launches"] == 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    # both arms print the SAME config object (the driver's same_config check): it is a module constant of bench.py
    assert d["config"] == _load_bench().CONFIG
    # --dump-outputs: the timed step's output dict, one float32 / float64 .npy per array
    assert all(p.suffix == ".npy" for p in dump.iterdir())
    arrays = {p.stem: np.load(p) for p in dump.iterdir()}
    assert {"dec_outputs", "wav_predictions", "log_duration_predictions"} <= set(arrays)
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    mel, wav = arrays["dec_outputs"], arrays["wav_predictions"]
    assert mel.dtype == np.float32 and mel.shape[0] == 1 and mel.shape[2] == 80 and wav.size == mel.shape[1] * 256
    assert np.isfinite(wav).all() and np.abs(wav).max() > 0


def test_headline_line_is_one_parsable_line_under_4k_even_when_sub_blocks_are_huge(capsys):
    """Round 1 lost its headline because a multi-KB 'experiments' object was embedded in the one JSON line.  `emit` is the
    only place that prints the line: it must stay < 4 KB (dropping optional sub-objects, never the contract keys), be the
    LAST stdout line, and send the long form elsewhere."""
    bench = _load_bench()
    line = {"metric": "mel_frames_per_sec", "value": 1.0, "unit": "mel-frames/s", "n_gpus": 1, "steps": 20, "warmup": 5,
            "ms_per_step": 1.0, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": bench.CONFIG, "e2e": {"value": 1.0, "unit": "mel-frames/s", "h2d_bytes_per_step": 1, "d2h_bytes_per_step": 1},
            "gpu_launches": 1, "roofline": {"bound": "tensor", "achieved": 1.0, "peak": 2.0, "unit": "TFLOP/s", "frac": 0.5, "traffic": None},
            "cpu_baseline": {"value": 1.0, "unit": "mel-frames/s", "cores": 1, "kind": "port", "sample": "x"},
            "clocks": {"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "reasons": []},
            "voc": {"k%d" % i: "x" * 200 for i in range(20)}, "cfg5": {"log": ["y" * 300] * 30}, "b32": {"ok": 1}}
    detail = {"long": ["z" * 1000] * 50}
    bench.emit(line, detail=detail)
    cap = capsys.readouterr()
    out = cap.out.splitlines()
    assert len(out) == 1 and len(out[0]) < 4096
    d = json.loads(out[0])
    _check_common(d)
    assert {"roofline", "cpu_baseline", "clocks"} <= set(d) and d["b32"] == {"ok": 1}
    assert "dropped" in d["cfg5"] and "dropped" in d["voc"]
    err = [l for l in cap.err.splitlines() if l.startswith("[bench detail] ")]
    assert len(err) == 1 and json.loads(err[0][len("[bench detail] "):]) == detail


def test_embedded_child_scripts_and_gpu_only_tools_compile():
    """Scripts that only ever run on the GPU box (child processes of the late GPU tests, the profiling tools, the checklist)
    must at least parse here: a syntax error there would cost a GPU call to find."""
    import ast
    import importlib.util
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("late_gpu_tests", os.path.join(root, "tests", "test_zz_late_round1_gpu.py"))
    src = open(spec.origin).read()
    tree = ast.parse(src)
    children = [n for n in tree.body if isinstance(n, ast.Assign) and isinstance(n.value, ast.Constant) and isinstance(n.value.value, str)
                and n.targets[0].id.endswith("_CHILD")]
    assert len(children) >= 1
    for n in children:
        compile(n.value.value, n.targets[0].id, "exec")
    for tool in sorted(os.listdir(os.path.join(root, "tools"))):
        path = os.path.join(root, "tools", tool)
        if tool.endswith(".py"):
            ast.parse(open(path).read(), filename=tool)
        elif tool.endswith(".sh"):
            assert subprocess.run(["bash", "-n", path]).returncode == 0, tool


def _unbound_names(src, fname="<src>"):
    import ast
    import builtins
    tree = ast.parse(src, fname)
    bound = set(dir(builtins))
    for n in ast.walk(tree):
        if isinstance(n, (ast.FunctionDef, ast.AsyncFunctionDef, ast.ClassDef)):
            bound.add(n.name)
            if not isinstance(n, ast.ClassDef):
                a = n.args
                for x in a.args + a.kwonlyargs + a.posonlyargs: bound.add(x.arg)
                if a.vararg: bound.add(a.vararg.arg)
                if a.kwarg: bound.add(a.kwarg.arg)
        elif isinstance(n, ast.Lambda):
            a = n.args
            for x in a.args + a.kwonlyargs + a.posonlyargs: bound.add(x.arg)
            if a.vararg: bound.add(a.vararg.arg)
            if a.kwarg: bound.add(a.kwarg.arg)
        elif isinstance(n, ast.Import):
            for al in n.names: bound.add((al.asname or al.name).split(".")[0])
        elif isinstance(n, ast.ImportFrom):
            for al in n.names: bound.add(al.asname or al.name)
        elif isinstance(n, ast.Name) and isinstance(n.ctx, (ast.Store, ast.Del)):
            bound.add(n.id)
        elif isinstance(n, ast.ExceptHandler) and n.name:
            bound.add(n.name)
        elif isinstance(n, ast.Global):
            bound.update(n.names)
    bad = sorted({n.id for n in ast.walk(tree) if isinstance(n, ast.Name) and isinstance(n.ctx, ast.Load) and n.id not in bound})
    return bad


def test_no_unbound_names_in_code_that_only_runs_on_the_gpu_box():
    """A crude static scan (every loaded name must be bound somewhere in its module): catches typos in the tools, the child
    scripts of the late GPU tests and the GPU-only branches of bench.py without a GPU."""
    import ast
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = [os.path.join(root, "bench.py"), os.path.join(root, "__graft_entry__.py")]
    for d in ("tools", "emotivoice_b200", "tests"):
        files += [os.path.join(root, d, f) for f in sorted(os.listdir(os.path.join(root, d))) if f.endswith(".py")]
    for f in files:
        assert [n for n in _unbound_names(open(f).read(), f) if n != "__file__"] == [], f
    late = ast.parse(open(os.path.join(root, "tests", "test_zz_late_round1_gpu.py")).read())
    for n in late.body:
        if isinstance(n, ast.Assign) and isinstance(n.value, ast.Constant) and isinstance(n.value.value, str) and n.targets[0].id.endswith("_CHILD"):
            assert _unbound_names(n.value.value) == [], n.targets[0].id
