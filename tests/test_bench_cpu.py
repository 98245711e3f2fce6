"""bench.py's reference arm (the reference's CPU reconcile loop, restated) runs without a GPU and
prints the one-line JSON contract the driver parses."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _line(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_reference_arm_contract():
    j = _line("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert j["impl"] == "reference" and j["metric"] == "task_reconciles_per_s" and j["unit"] == "reconciles/s"
    assert j["higher_is_better"] is True and j["n_gpus"] == 1 and j["steps"] == 1 and j["warmup"] == 1
    assert j["value"] > 0 and j["ms_per_step"] > 0 and j["gpu_launches"] == 0
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == j["value"] and "sample" in cb
    assert j["e2e"] == {"value": j["value"], "unit": j["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "512 concurrent Task CRs" in j["config"]["workload"] and "window tokens per step" in j["config"]["workload"]


def test_reference_arm_never_maps_the_product_library():
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0', '--config', '1']\n"
            "runpy.run_path(%r, run_name='__main__')\n"
            "maps = open('/proc/self/maps').read()\n"
            "assert 'libacp_host.so' in maps and 'libacp_infer' not in maps, 'product library mapped by the reference arm'\n"
            % os.path.join(ROOT, "bench.py"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]


def test_dump_outputs_writes_fixed_width_byte_rows(tmp_path):
    code = ("import runpy, sys\n"
            "runpy.run_path(%r)['dump_outputs'](sys.argv[1], ['test', '', 'caf\\u00e9 ' * 3], 2)\n" % os.path.join(ROOT, "bench.py"))
    out = subprocess.run([sys.executable, "-c", code, str(tmp_path / "d")], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    import numpy as np
    a = np.load(tmp_path / "d" / "task_output_bytes.npy")
    assert a.dtype == np.float32 and a.shape == (3, 18)         # the third output is longer than 5 * max_tokens
    assert a[0, :4].tolist() == list(b"test") and (a[0, 4:] == -1).all() and (a[1] == -1).all()
    assert bytes(a[2].astype(np.uint8)) == "café café café ".encode()


def test_steps_and_dump_arguments_are_checked():
    for args in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "x"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                             timeout=120, cwd=ROOT)
        assert out.returncode == 2 and "error:" in out.stderr, (args, out.stderr[-500:])


def test_reference_arm_follows_the_config_flag():
    j = _line("--impl", "reference", "--config", "3", "--steps", "1", "--warmup", "0")
    assert j["impl"] == "reference" and "256 concurrent Task CRs" in j["config"]["workload"]
