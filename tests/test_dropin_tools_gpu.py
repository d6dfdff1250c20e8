"""Drop-in proof on the GPU: the reference's OWN tools (tools/benchmodel.cpp, tools/render.cpp,
tools/loadmodel.cpp), compiled unchanged against include/NAM/*.h + libnam_b200.so into oracle/_ref/tools/ by
`make -C oracle ref_tools` (build() runs it where the reference checkout is readable), run here and are
checked against the CPU oracle.  Also the repo's own C++ host tool over the C ABI.  The reference's tools are skipped
where they were not built: their sources are not part of this repository."""
import json
import struct
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import oracle
from tests import nam_fixtures as fx

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
REF_TOOLS = ROOT / "oracle" / "_ref" / "tools"


def _write_nam(tmp_path, name):
    p = tmp_path / f"{name}.nam"
    p.write_text(json.dumps(fx.load_model(name)))
    return p


def _write_wav24(path, x, rate=48000):
    v = np.clip(np.round(x.astype(np.float64) * 8388608.0), -8388608, 8388607).astype(np.int32)
    b = np.zeros((len(v), 3), np.uint8)
    b[:, 0], b[:, 1], b[:, 2] = v & 0xFF, (v >> 8) & 0xFF, (v >> 16) & 0xFF
    data = b.tobytes()
    hdr = b"RIFF" + struct.pack("<I", 36 + len(data)) + b"WAVE" + b"fmt " + struct.pack("<IHHIIHH", 16, 1, 1, rate, rate * 3, 3, 24)
    path.write_bytes(hdr + b"data" + struct.pack("<I", len(data)) + data)


def _read_wav_f32(path):
    d = path.read_bytes()
    assert d[:4] == b"RIFF" and d[8:12] == b"WAVE"
    pos = d.index(b"data") + 8
    return np.frombuffer(d[pos:], dtype="<f4")


def _need(binary):
    p = REF_TOOLS / binary
    if not p.exists():
        pytest.skip(f"{p} not built (reference tree absent at build time)")
    return p


@pytest.mark.parametrize("name", ["wavenet", "wavenet_a1_standard", "lstm"])
def test_reference_benchmodel_runs_unchanged(tmp_path, name):
    """tools/benchmodel.cpp: fast tanh on, Reset(sr, 64), 1500 x process(zeros, 64)."""
    exe = _need("benchmodel")
    for extra in ([], ["--no-fast-tanh"]):
        r = subprocess.run([str(exe), *extra, str(_write_nam(tmp_path, name))], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout + r.stderr
        assert "Finished" in r.stdout and r.stdout.strip().splitlines()[-1].endswith("ms")


def test_reference_loadmodel_and_errors(tmp_path):
    exe = _need("loadmodel")
    r = subprocess.run([str(exe), str(_write_nam(tmp_path, "wavenet"))], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "Model loaded successfully" in r.stderr
    r = subprocess.run([str(exe), str(tmp_path / "missing.nam")], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0  # NamFileValidationError propagates like in the reference


@pytest.mark.parametrize("name", ["wavenet", "wavenet_a1_standard", "lstm"])
def test_reference_render_matches_oracle(tmp_path, name):
    """tools/render.cpp: model + mono WAV -> float32 WAV in 64-frame blocks (exact tanh); compare with the oracle."""
    exe = _need("render")
    x = fx.input_wav()[40000:56000] if name == "wavenet_a1_standard" else fx.input_wav()[:30000]
    wav_in, wav_out = tmp_path / "in.wav", tmp_path / "out.wav"
    _write_wav24(wav_in, x)
    r = subprocess.run([str(exe), str(_write_nam(tmp_path, name)), str(wav_in), str(wav_out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    y = _read_wav_f32(wav_out)
    m = oracle.OracleModel.from_dict(fx.load_model(name))
    m.reset(48000.0, 64)
    ref = m.run(x, 64)
    assert len(y) == len(ref)
    assert np.max(np.abs(y - ref)) <= 1e-5


def test_own_cxx_tool_over_the_c_abi(tmp_path):
    exe = ROOT / "build" / "nam_b200_bench"
    if not exe.exists():
        pytest.skip("build/nam_b200_bench not built")
    r = subprocess.run([str(exe), "--batch", "64", "--frames", "256", "--calls", "20", str(_write_nam(tmp_path, "wavenet_a1_standard"))],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["batch"] == 64 and out["msamples_per_s"] > 0 and np.isfinite(out["last_output"])


def test_reference_tools_on_a_slimmable_container(tmp_path):
    """tools/benchmodel.cpp --slim / tools/render.cpp --slim dynamic_cast the model to nam::SlimmableModel
    (benchmodel.cpp:93-100): a SlimmableContainer file must load as one, a plain model must be refused."""
    exe = _need("benchmodel")
    cont = tmp_path / "a2.nam"
    cont.write_text(json.dumps(fx.make_container([(0.5, fx.load_model("a2_lite")), (1.0, fx.load_model("a2_full"))])))
    r = subprocess.run([str(exe), str(cont), "--slim", "0.25"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Setting slimmable size to 0.25" in r.stdout and "Finished" in r.stdout
    r = subprocess.run([str(exe), str(_write_nam(tmp_path, "wavenet")), "--slim", "0.25"], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode != 0 and "SlimmableModel" in (r.stdout + r.stderr)
    # render through the container at the small size == the oracle of the small model
    rexe = _need("render")
    x = fx.input_wav()[44000:52000]
    wav_in, wav_out = tmp_path / "in.wav", tmp_path / "out.wav"
    _write_wav24(wav_in, x)
    r = subprocess.run([str(rexe), str(cont), str(wav_in), str(wav_out), "--slim", "0.25"], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    m = oracle.OracleModel.from_dict(fx.load_model("a2_lite"))
    m.reset(48000.0, 64)
    assert np.max(np.abs(_read_wav_f32(wav_out) - m.run(x, 64))) <= 1e-5


@pytest.mark.parametrize("bufsize", [16, 64, 512])
def test_reference_benchmodel_bufsize_runs_unchanged(tmp_path, bufsize):
    """tools/benchmodel_bufsize.cpp:19-110: model, buffer size, iterations -> one CSV line 'bufsize,avg_microseconds'."""
    exe = _need("benchmodel_bufsize")
    r = subprocess.run([str(exe), str(_write_nam(tmp_path, "wavenet_a1_standard")), str(bufsize), "50"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    b, us = r.stdout.strip().splitlines()[-1].split(",")
    assert int(b) == bufsize and float(us) > 0.0


def test_cpp_host_drives_several_gpus_through_the_c_abi(tmp_path):
    """tools/nam_b200_multi_test.cpp: nam_b200_multi_* (one worker thread + one complete handle per GPU, the batch dealt out
    in contiguous shards) reproduces a single-device handle bit for bit.  With one GPU visible the same device is listed
    twice (two handles, two worker threads on one GPU); with two or more, devices 0 and 1."""
    import torch

    exe = ROOT / "build" / "nam_b200_multi_test"
    if not exe.exists():
        pytest.skip(f"{exe} not built")
    devs = ["0", "1"] if torch.cuda.device_count() >= 2 else ["0", "0"]
    r = subprocess.run([str(exe), str(_write_nam(tmp_path, "wavenet_a1_standard")), "600", "2048", *devs],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "bit-identical" in r.stdout, r.stdout
