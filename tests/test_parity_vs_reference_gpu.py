"""The CUDA path against THE REFERENCE ITSELF (the unmodified NeuralAmpModelerCore sources compiled against
oracle/eigen_shim, see tests/test_reference_build.py; its outputs are recorded in tests/golden/reference_outputs.npz),
through the C ABI, 1e-5 max-abs on the recorded frames."""
import numpy as np
import pytest

import neuralampmodelercore_b200 as nb
from tests import nam_fixtures as fx
from tests import reference_outputs as R

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _gpu(nam, x, fast, block, **kw):
    d = nb.get_dsp(nam, batch=1, fast_tanh=fast, **kw)
    d.Reset(48000.0, block)
    y = np.concatenate([d.process_batch(np.ascontiguousarray(x[None, p:p + block]))[0] for p in range(0, len(x), block)])
    d.close()
    return y


@pytest.mark.parametrize("name", ["wavenet", "wavenet_a1_standard", "a2_lite", "a2_full", "wavenet_condition_dsp",
                                  "wavenet_a2_max"])
@pytest.mark.parametrize("fast", [False, True], ids=["exact_tanh", "fast_tanh"])
def test_wavenets_match_the_reference(name, fast):
    nam = fx.load_model(name)
    x = fx.input_wav()[43000:53000]
    yr = R.expected(f"wav/{name}/{R.regime(fast)}")["y"]
    for block in (64, 4096):  # the tools' block size and one big call
        err = float(np.max(np.abs(R.sample(_gpu(nam, x, fast, block)) - yr)))
        assert err / max(1.0, float(np.max(np.abs(yr)))) <= TOL, f"{name} block {block}: {err:.3e}"


@pytest.mark.parametrize("fast", [False, True], ids=["exact_tanh", "fast_tanh"])
def test_lstm_matches_the_reference(fast):
    nam = fx.load_model("lstm")
    x = fx.input_wav()[43000:53000]
    # prewarm rounds up to whole 64-frame blocks (lstm.cpp:127-134): same block here
    yr = R.expected(f"wav/lstm/{R.regime(fast)}")["y"]
    err = float(np.max(np.abs(R.sample(_gpu(nam, x, fast, 64)) - yr)))
    assert err <= TOL, f"{err:.3e}"


def test_tensor_core_and_general_kernels_match_the_reference():
    nam = fx.load_model("wavenet_a1_standard")
    x = fx.input_wav()[45000:51000]
    yr = R.expected("wav_45000/wavenet_a1_standard/exact")["y"]
    # (kernel_geometry 3 = the tensor-core kernel, a build option: NAM_B200_BUILD_TC=1)
    for geom in (1, 2, 3, 4) if nb.has_tensor_core_kernel() else (1, 2, 4):
        err = float(np.max(np.abs(R.sample(_gpu(nam, x, False, 2048, kernel_geometry=geom)) - yr)))
        assert err <= TOL, f"kernel_geometry {geom}: {err:.3e}"


def test_container_matches_the_reference():
    cont = fx.make_container([(0.5, fx.load_model("a2_lite")), (1.0, fx.load_model("a2_full"))])
    x = fx.synthetic_batch(1, 3000, seed=31)[0]
    for slim in (None, 0.3):
        yr = R.expected(f"container/{slim}")["y"]
        d = nb.get_dsp(cont, batch=1)
        if slim is not None:
            d.SetSlimmableSize(slim)
        d.Reset(48000.0, 1000)
        y = np.concatenate([d.process_batch(np.ascontiguousarray(x[None, p:p + 1000]))[0] for p in range(0, 3000, 1000)])
        d.close()
        assert float(np.max(np.abs(R.sample(y) - yr))) <= TOL, f"slim {slim}"


def test_second_reset_and_standalone_prewarm_follow_the_reference():
    """DSP::Reset = SetMaxBufferSize + prewarm (NAM/dsp.cpp:130-140).  The reference's LSTM overrides neither Reset nor
    SetMaxBufferSize, so its hidden / cell state survives a Reset and only the prewarm runs on top of it; the WaveNet's
    ring buffers are cleared.  Audio, Reset, audio again -- and a standalone prewarm() in the middle of a stream -- against the
    reference build doing the same."""
    x = fx.synthetic_batch(1, 3 * 1024, seed=17)[0]
    for name in ("lstm", "wavenet"):
        nam = fx.load_model(name)
        d = nb.get_dsp(nam, batch=3, fast_tanh=False)
        d.Reset(48000.0, 64)
        got = []
        for part in range(3):
            seg = x[part * 1024:(part + 1) * 1024]
            # three streams with different gains: they diverge, so the later prewarms must run on every stream
            xb = np.ascontiguousarray(np.stack([seg, 0.5 * seg, -seg]))
            got.append(np.concatenate([d.process_batch(np.ascontiguousarray(xb[:, p:p + 64])) for p in range(0, 1024, 64)], axis=1)[0])
            if part == 0:
                d.Reset(48000.0, 64)
            elif part == 1:
                d.prewarm()
        d.close()
        want = R.expected(f"reset_prewarm/{name}")["y"]
        err = float(np.max(np.abs(R.sample(np.concatenate(got)) - want)))
        assert err <= TOL, f"{name}: {err:.3e}"
