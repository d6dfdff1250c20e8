"""Whole-model pin of the oracle against THE REFERENCE ITSELF: the unmodified NeuralAmpModelerCore source tree compiled
against a stand-in for its missing Eigen submodule (oracle/eigen_shim, recipe `make -C oracle ref`), whose outputs
are recorded in tests/golden/reference_outputs.npz (tests/reference_outputs.py).  The reference's own tests hold no
whole-model vectors (SURVEY.md 8c), so this is what turns the oracle's model-level reading of the reference -- weight
order, prewarm, head_scale, condition_dsp, containers, the A2 fast path -- from "restated" into "checked".

Runs on CPU."""
import numpy as np
import pytest

from oracle import oracle, ref
from tests import nam_fixtures as fx
from tests import reference_outputs as R

# two independent fp32 implementations (different summation order inside the matrix products): the reference's
# authors accept 5e-5 between two of their own (tools/test/test_a2_fast.cpp:296-298); measured here <= 3e-6
TOL = 1e-5

MODELS = ["wavenet", "wavenet_a1_standard", "lstm", "wavenet_condition_dsp", "wavenet_a2_max", "a2_lite", "a2_full"]


def _rel(err, y):
    return err / max(1.0, float(np.max(np.abs(y))))


def _oracle(nam, x, block=64, fast=False):
    m = oracle.OracleModel.from_dict(nam, fast_tanh=fast)
    m.reset(48000.0, block)
    return m.run(x, block)


@pytest.mark.parametrize("name", MODELS)
@pytest.mark.parametrize("fast", [False, True], ids=["exact_tanh", "fast_tanh"])
def test_oracle_matches_the_reference_build(name, fast):
    nam = fx.load_model(name)
    x = fx.input_wav()[43000:53000]  # 5,000 frames of silence, then the 220 Hz sine
    want = R.expected(f"wav/{name}/{R.regime(fast)}")
    m = oracle.OracleModel.from_dict(nam, fast_tanh=fast)
    m.reset(48000.0, 64)
    assert want["prewarm_samples"] == m.prewarm_samples
    yr, yo = want["y"], R.sample(m.run(x, 64))
    err = float(np.max(np.abs(yr - yo)))
    assert _rel(err, yr) <= TOL, f"{name}: max|reference - oracle| = {err:.3e} (max|y| {np.max(np.abs(yr)):.3f})"


@pytest.mark.parametrize("name", ["wavenet_a1_standard", "a2_full", "lstm"])
def test_block_size_protocols_agree(name):
    """The reference at maxBufferSize 64 (tools) vs 1000: same stream (prewarmed WaveNet state is block-size
    independent; the LSTM prewarm rounds up to whole blocks, lstm.cpp:127-134, so compare like with like)."""
    nam = fx.load_model(name)
    x = fx.synthetic_batch(1, 3000, seed=17)[0]
    for block in (64, 1000):
        yr = R.expected(f"blocks/{name}/{block}")["y"]
        yo = R.sample(_oracle(nam, x, block))
        assert _rel(float(np.max(np.abs(yr - yo))), yr) <= TOL, f"{name} block {block}"


def test_golden_vectors_were_not_a_misreading():
    """The committed oracle vectors (tests/golden/oracle_outputs.npz) against the reference build, full 2 s."""
    for name in ("wavenet", "wavenet_a1_standard", "a2_full"):
        gold = fx.oracle_golden(name, "exact")
        for key, val in R.expected(f"full_input/{name}").items():
            assert np.max(np.abs(val - R.sample(gold[key]))) <= TOL, f"{name} {key}"


def test_a2_fast_path_and_generic_path_of_the_reference():
    """The default reference build routes A2 shapes to A2FastModel (model.cpp:1317-1320); the second build has the
    fast path compiled out.  Both must agree with the oracle (and so with each other)."""
    x = fx.synthetic_batch(1, 4000, seed=3)[0]
    for name in ("a2_lite", "a2_full"):
        yo = R.sample(_oracle(fx.load_model(name), x))
        for variant in ("default", "generic"):
            err = float(np.max(np.abs(R.expected(f"a2_variants/{name}/{variant}")["y"] - yo)))
            assert err <= TOL, f"{name} {variant}: {err:.3e}"


def test_slimmable_container_semantics():
    """ContainerModel (container.cpp): full size by default; SetSlimmableSize before or after Reset; the newly
    active sub-model starts from its own prewarmed state."""
    lite, full = fx.load_model("a2_lite"), fx.load_model("a2_full")
    x = fx.synthetic_batch(1, 2000, seed=9)[0]
    want = R.expected("container_semantics")

    def orc(nam, sig):
        return R.sample(_oracle(nam, sig))

    assert np.max(np.abs(want["full_first"] - orc(full, x[:1000]))) <= TOL
    assert np.max(np.abs(want["small"] - orc(lite, x))) <= TOL  # SetSlimmableSize(0.2)
    assert np.max(np.abs(want["full_again"] - orc(full, x[:640]))) <= TOL  # 0.5 is not < 0.5 -> full again, freshly reset
    # SetSlimmableSize(0.1) before the first Reset (tools/render.cpp:117-126 order)
    assert np.max(np.abs(want["small_before_reset"] - orc(lite, x))) <= TOL


def _multichannel_models():
    from oracle import nam_config

    def rnd(nam, seed, last=None):
        n = nam_config.expected_weight_count(nam)
        w = np.random.default_rng(seed).uniform(-0.35, 0.35, size=n).astype(np.float32)
        if last is not None:
            w[-1] = last
        nam["weights"] = [float(v) for v in w]
        return nam

    a0 = {"input_size": 2, "condition_size": 2, "head_size": 4, "channels": 5, "kernel_size": 3, "dilations": [1, 2, 4, 9],
          "activation": "Tanh", "gated": False, "head_bias": False}
    a1 = {"input_size": 5, "condition_size": 2, "head_size": 3, "channels": 4, "kernel_size": 3, "dilations": [1, 6],
          "activation": "Tanh", "gated": True, "head_bias": True}
    yield "wavenet 2 in / 3 out", rnd(fx.make_wavenet_nam([a0, a1], [], head_scale=0.5, in_channels=2), 4, last=0.5)
    for ci, co, H, nl in ((2, 3, 5, 1), (3, 1, 8, 2)):
        nam = {"version": "0.5.4", "architecture": "LSTM", "sample_rate": 48000.0,
               "config": {"in_channels": ci, "out_channels": co, "input_size": ci, "hidden_size": H, "num_layers": nl},
               "weights": []}
        yield f"lstm {ci} in / {co} out", rnd(nam, ci * 10 + co)


def _planar_against_the_reference(nam, fast, n, block, seed, key, label=""):
    """Multi-channel DSP::process calls of `block` frames on synthetic input, the oracle against the recorded run."""
    want = R.expected(key)
    o = oracle.OracleModel.from_dict(nam, fast_tanh=fast)
    assert (want["in_channels"], want["out_channels"], want["prewarm_samples"]) == (
        o.in_channels, o.out_channels, o.prewarm_samples), label
    o.reset(48000.0, block)
    x = fx.synthetic_batch(o.in_channels, n, seed=seed)
    yo = np.concatenate([np.atleast_2d(o.process(np.ascontiguousarray(x[:, p:p + block]))) for p in range(0, n, block)],
                        axis=1)
    o.close()
    err = np.max(np.abs(want["y"] - R.sample(yo)), axis=0)  # per sampled frame, over the channels
    assert float(err.max()) <= TOL, f"{label} block at {int(np.argmax(err)) * R.STRIDE // block * block}: {err.max():.3e}"


def test_multichannel_models():
    """in_channels / out_channels != 1 (NAM/wavenet/model.cpp:809-820,888-909; NAM/lstm.cpp:103-125): the oracle's
    reading of the channel handling against the reference build, DSP::process with channel arrays."""
    for i, (label, nam) in enumerate(_multichannel_models()):
        _planar_against_the_reference(nam, False, 640, 64, 17, f"multichannel/{i}", label)


def _convnet(channels, dilations, batchnorm, activation, seed, in_channels=1, out_channels=1, groups=1):
    from oracle import nam_config

    nam = {"version": "0.5.4", "architecture": "ConvNet", "sample_rate": 48000.0,
           "config": {"channels": channels, "dilations": list(dilations), "batchnorm": batchnorm, "activation": activation,
                      "groups": groups, "in_channels": in_channels, "out_channels": out_channels},
           "weights": []}
    n = nam_config.expected_weight_count(nam)
    rng = np.random.default_rng(seed)
    w = rng.uniform(-0.4, 0.4, size=n).astype(np.float32)
    if batchnorm:  # running_var and eps must be positive (convnet.cpp:34): walk the stream like the constructor does
        pos, cin = 0, in_channels
        for _d in dilations:
            pos += (cin * channels * 2) // groups
            w[pos + channels:pos + 2 * channels] = rng.uniform(0.5, 1.5, size=channels)
            w[pos + 4 * channels] = 1e-5
            pos += 4 * channels + 1
            cin = channels
    nam["weights"] = [float(v) for v in w]
    return nam


CONVNETS = [
    dict(channels=8, dilations=[1, 2, 4, 8, 16, 32], batchnorm=True, activation="Tanh", seed=1),
    dict(channels=5, dilations=[1, 3, 9], batchnorm=False, activation="ReLU", seed=2),
    dict(channels=6, dilations=[2, 4, 64, 128], batchnorm=True, activation={"type": "LeakyReLU", "negative_slope": 0.05},
         seed=3, in_channels=2, out_channels=3, groups=1),
    dict(channels=4, dilations=[1, 2], batchnorm=False, activation="Sigmoid", seed=4, groups=2, in_channels=2),
]


@pytest.mark.parametrize("kw", CONVNETS, ids=[f"convnet{i}" for i in range(len(CONVNETS))])
@pytest.mark.parametrize("fast", [False, True], ids=["exact_tanh", "fast_tanh"])
def test_convnet(kw, fast):
    """NAM/convnet.cpp (kernel-2 dilated Conv1D -> BatchNorm -> activation blocks, linear head): the reference's own
    tests only assert isfinite (tools/test/test_convnet.cpp), so the oracle's reading is held to the reference build."""
    _planar_against_the_reference(_convnet(**kw), fast, 960, 96, 23, f"convnet/{CONVNETS.index(kw)}/{R.regime(fast)}")


def _slimmable_models():
    """(label, nam) pairs: the reference's own example and a two-array model that exercises every slicing rule of
    NAM/wavenet/slimmable.cpp:133-262 (gated conv, bottleneck != channels, head1x1, FiLM with and without shift)."""
    from oracle import nam_config

    yield "example_models/slimmable_wavenet.nam", fx.load_model("slimmable_wavenet")

    def film(active=True, shift=True):
        return {"active": active, "shift": shift, "groups": 1}

    slim = lambda allowed: {"method": "slice_channels_uniform", "kwargs": {"allowed_channels": allowed}}  # noqa: E731
    a0 = {"input_size": 1, "condition_size": 1, "channels": 6, "bottleneck": 4, "head_size": 4, "head_bias": False,
          "kernel_sizes": [3, 2, 3], "dilations": [1, 2, 5], "activation": "Tanh",
          "gating_mode": ["gated", "none", "blended"], "secondary_activation": ["Sigmoid", "Sigmoid", "Sigmoid"],
          "layer1x1": {"active": True, "groups": 1}, "head1x1": {"active": True, "out_channels": 5, "groups": 1},
          "conv_pre_film": film(), "conv_post_film": film(shift=False), "input_mixin_pre_film": film(),
          "activation_post_film": film(), "layer1x1_post_film": film(shift=False), "head1x1_post_film": film(),
          "slimmable": slim([2, 4, 6])}
    a1 = {"input_size": 6, "condition_size": 1, "channels": 4, "head_size": 1, "head_bias": True, "kernel_size": 3,
          "dilations": [1, 4], "activation": "ReLU", "gating_mode": "none", "slimmable": slim([1, 4])}
    nam = fx.make_wavenet_nam([a0, a1], [], head_scale=0.3, version="0.7.0")
    nam["config"]["layers"][0]["head_size"] = 4  # feeds array 1 (channels 4)
    n = nam_config.expected_weight_count(nam)
    w = np.random.default_rng(77).uniform(-0.4, 0.4, size=n).astype(np.float32)
    w[-1] = 0.3
    nam["weights"] = [float(v) for v in w]
    yield "two arrays, gated / blended, head1x1, FiLM", nam


@pytest.mark.parametrize("case", [0, 1])
def test_slimmable_wavenet_slicing(case):
    """A WaveNet with "slimmable" layer arrays is a SlimmableWavenet in the reference (model.cpp:1290-1315): the PRODUCT's
    loader turns it into one sliced plain WaveNet per ratio interval (nam_b200_submodel_json, host only).  Every such
    document, run by the oracle, must equal the reference build after SetSlimmableSize(ratio) -- at interval midpoints,
    at the breakpoints themselves and at 0 / 1."""
    import neuralampmodelercore_b200 as nb

    label, nam = list(_slimmable_models())[case]
    subs = nb.submodels(nam)
    assert len(subs) >= 2 and subs[-1][0] >= 1.0
    want = R.expected(f"slimmable/{case}")
    ratios = R.slimmable_ratios(subs)
    assert np.array_equal(want["ratios"], ratios), f"{label}: the sub-model breakpoints moved: {ratios}"
    x = fx.synthetic_batch(1, 1500, seed=41)[0]
    for val, yr in zip(ratios, want["y"]):
        idx = next((i for i, (mv, _) in enumerate(subs) if val < mv), len(subs) - 1)
        yo = R.sample(_oracle(subs[idx][1], x))
        assert _rel(float(np.max(np.abs(yr - yo))), yr) <= TOL, f"{label}: ratio {val} -> sub-model {idx}"


@pytest.mark.parametrize("impl", ["direct", "fft", "auto"])
def test_linear_fft_and_direct_form_are_the_same_filter(impl):
    """NAM/linear.cpp:99-113,201-278: above 256 taps the reference's Linear switches ("auto") or can be told ("fft") to a
    partitioned-FFT evaluation of the same FIR.  The product runs direct form at any length (SURVEY.md 8f-4), so the two
    must agree: the reference build with each implementation against the oracle's direct form."""
    x = fx.synthetic_batch(1, 3000, seed=5)[0]
    want = R.sample(_oracle(linear_fir(impl), x))
    got = R.expected(f"linear/{impl}")["y"]
    assert float(np.max(np.abs(got - want))) <= 2e-6


def linear_fir(impl):
    """A 600-tap Linear model (past the reference's 256-tap switch to FFT) with the given "implementation"."""
    rng = np.random.default_rng(12)
    rf = 600
    return {"version": "0.5.4", "architecture": "Linear", "sample_rate": 48000,
            "config": {"receptive_field": rf, "bias": True, "implementation": impl},
            "weights": [float(v) for v in rng.uniform(-0.05, 0.05, rf + 1)]}


@pytest.mark.skipif(not (ref.available() and ref.available("generic")), reason="oracle/_ref/ not built")
def test_recorded_outputs_are_the_reference_builds():
    """tests/golden/reference_outputs.npz is what the reference build computes: every recorded run, repeated."""
    with np.load(R.GOLDEN) as z:
        stored = {k: z[k] for k in z.files}
    fresh = R.record()
    assert sorted(fresh) == sorted(stored)
    for key, val in fresh.items():
        assert val.shape == stored[key].shape and float(np.max(np.abs(val - stored[key]), initial=0.0)) <= 1e-6, key
