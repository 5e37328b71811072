"""bench.py host logic that can run without a GPU: the reference (CPU) arm and its isolation from the product."""
import json
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_runs_the_reference_and_never_maps_the_product_library():
    """`bench.py --impl reference` must time the reference's own code (kind "reference" when tools/ref_import.py finds a
    copy of the reference, else the oracle port) and must not dlopen libstylesinger_b200.so (an earlier arm imported
    stylesinger_b200.dist -> engine -> _lib)."""
    code = (
        "import sys, json, io, contextlib\n"
        f"sys.path.insert(0, {REPO!r}); sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '1', '--T', '2', "
        "'--cpu-sample-seconds', '0.3']\n"
        "import bench\n"
        "buf = io.StringIO()\n"
        "with contextlib.redirect_stdout(buf):\n"
        "    bench.main()\n"
        "line = [l for l in buf.getvalue().splitlines() if l.startswith('{')][-1]\n"
        "maps = open('/proc/self/maps').read()\n"
        "print('RESULT ' + json.dumps({'line': json.loads(line), 'mapped': 'libstylesinger_b200' in maps}))\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900, cwd=REPO)
    assert r.returncode == 0, r.stderr[-2000:]
    res = json.loads([l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1][7:])
    assert res["mapped"] is False
    line = res["line"]
    assert line["impl"] == "reference" and line["gpu_launches"] == 0 and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port")
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    sys.path.insert(0, os.path.join(REPO, "tools"))
    import ref_import
    assert line["cpu_baseline"]["kind"] == ("reference" if ref_import.find_reference() is not None else "port")


def test_dump_outputs_keeps_within_the_budget_with_a_fixed_row_sample(tmp_path, monkeypatch):
    import numpy as np
    import torch
    sys.path.insert(0, REPO)
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    g = torch.Generator().manual_seed(0)
    arrays = {"mel_out": torch.randn(6000, 80, generator=g), "wav": torch.randn(6000, 256, generator=g),
              "wav_frame_offsets": np.array([0, 2500, 6000], np.int32)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    total = sum(f.stat().st_size for f in (tmp_path / "a").iterdir())
    assert total <= (1 << 20) + 4096, total
    offs = np.load(tmp_path / "a" / "wav_frame_offsets.npy")
    assert offs.dtype == np.float64 and np.array_equal(offs, [0, 2500, 6000])
    rows = np.load(tmp_path / "a" / "mel_out_rows.npy").astype(np.int64)
    assert np.array_equal(rows, np.load(tmp_path / "b" / "wav_rows.npy"))  # same seeded rows, run to run and array to array
    mel = np.load(tmp_path / "a" / "mel_out.npy")
    assert mel.dtype == np.float32 and np.array_equal(mel, arrays["mel_out"].numpy()[rows])
    for extra in (["--impl", "reference"], ["--workload", "sweep"], ["--steps", "0"]):  # refused before any work starts
        monkeypatch.setattr(sys, "argv", ["bench.py", "--dump-outputs", str(tmp_path / "c")] + extra)
        with pytest.raises(SystemExit) as e:
            bench.main()
        assert e.value.code == 2 and not (tmp_path / "c").exists()
