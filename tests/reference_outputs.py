"""Outputs of the reference itself (NeuralAmpModelerCore, built into oracle/_ref/ by `make -C oracle ref`), recorded
in tests/golden/reference_outputs.npz so that the comparisons with it run on every machine, with or without the
reference's sources.

_runs() names every reference run the suite compares with; each returns the arrays the tests read, the signals already
passed through sample().  The tests compare sample() of their own outputs with them.  Re-record after changing a run:

    python -c "import __graft_entry__ as g; g.build()"    # NAM_REFERENCE=<checkout> if not oracle/Makefile's REF
    python -m tests.reference_outputs
"""
from __future__ import annotations

import functools

import numpy as np

from tests import nam_fixtures as fx

GOLDEN = fx.GOLDEN / "reference_outputs.npz"
# every 7th frame: coprime with every block size the tests use, so each position inside a block is checked
STRIDE = 7


def sample(y: np.ndarray) -> np.ndarray:
    """The frames of a signal (last axis) that are stored."""
    return np.ascontiguousarray(np.asarray(y)[..., ::STRIDE])


def regime(fast: bool) -> str:
    return "fast" if fast else "exact"


@functools.lru_cache(maxsize=None)
def _stored() -> dict:
    with np.load(GOLDEN) as z:
        return {k: z[k] for k in z.files}


def expected(key: str) -> dict:
    """The recorded arrays of run `key`."""
    out = {k.split("/")[-1]: v for k, v in _stored().items() if k.rsplit("/", 1)[0] == key}
    assert out, f"{key}: not recorded in {GOLDEN.name} (python -m tests.reference_outputs)"
    return out


# ---------------------------------------------------------------------------------------------------------------------
# The runs, on the reference build (oracle.ref).  Each mirrors the reference side of the test that reads it.

def _model(nam, fast=False, variant="default"):
    from oracle import ref

    return ref.ReferenceModel.from_dict(nam, fast_tanh=fast, variant=variant)


def _stream(nam, x, fast=False, block=64, slim=None, variant="default"):
    """get_dsp, [SetSlimmableSize,] Reset(48 kHz, block), `block`-frame process() calls."""
    r = _model(nam, fast, variant)
    if slim is not None:
        r.set_slimmable_size(slim)
    r.reset(48000.0, block)
    out = {"y": sample(r.run(x, block)), "prewarm_samples": np.int64(r.prewarm_samples)}
    r.close()
    return out


def _planar(nam, fast, n, block, seed):
    """Multi-channel DSP::process calls on synthetic input (in_channels, n) in `block`-frame calls."""
    r = _model(nam, fast)
    r.reset(48000.0, block)
    x = fx.synthetic_batch(r.in_channels, n, seed=seed)
    y = np.concatenate([r.process_planar(x[:, p:p + block]) for p in range(0, n, block)], axis=1)
    out = {"y": sample(y), "in_channels": np.int64(r.in_channels), "out_channels": np.int64(r.out_channels),
           "prewarm_samples": np.int64(r.prewarm_samples)}
    r.close()
    return out


def _full_input_decimated(name):
    r = _model(fx.load_model(name))
    r.reset(48000.0, 64)
    y = r.run(fx.input_wav(), 64)
    r.close()
    return {k: sample(v) for k, v in fx.decimate(y).items()}


def _container_semantics():
    lite, full = fx.load_model("a2_lite"), fx.load_model("a2_full")
    cont = fx.make_container([(0.5, lite), (1.0, full)])
    x = fx.synthetic_batch(1, 2000, seed=9)[0]
    r = _model(cont)
    r.reset(48000.0, 64)
    out = {"full_first": sample(r.run(x[:1000], 64))}
    r.set_slimmable_size(0.2)
    out["small"] = sample(r.run(x, 64))
    r.set_slimmable_size(0.5)
    out["full_again"] = sample(r.run(x[:640], 64))
    r.close()
    r = _model(cont)
    r.set_slimmable_size(0.1)
    r.reset(48000.0, 64)
    out["small_before_reset"] = sample(r.run(x, 64))
    r.close()
    return out


def slimmable_ratios(subs) -> list[float]:
    """0, 1, every breakpoint of the product's sub-model list and the midpoints between them."""
    bps = [mv for mv, _ in subs[:-1]]
    return sorted({0.0, 1.0, *bps, *[(a + b) / 2 for a, b in zip([0.0] + bps, bps + [1.0])]})


def _slimmable(case):
    import neuralampmodelercore_b200 as nb
    from tests.test_reference_build import _slimmable_models

    _, nam = list(_slimmable_models())[case]
    ratios = slimmable_ratios(nb.submodels(nam))
    x = fx.synthetic_batch(1, 1500, seed=41)[0]
    ys = []
    for val in ratios:
        r = _model(nam)
        r.reset(48000.0, 64)
        r.set_slimmable_size(val)
        ys.append(r.run(x, 64))
        r.close()
    return {"ratios": np.asarray(ratios), "y": sample(np.stack(ys))}


def _reset_and_prewarm(name):
    """Audio, Reset, audio, standalone prewarm(), audio: 3 x 1024 frames in 64-frame calls."""
    x = fx.synthetic_batch(1, 3 * 1024, seed=17)[0]
    r = _model(fx.load_model(name))
    r.reset(48000.0, 64)
    want = []
    for part in range(3):
        want.append(r.run(x[part * 1024:(part + 1) * 1024], 64))
        if part == 0:
            r.reset(48000.0, 64)
        elif part == 1:
            r.prewarm()
    r.close()
    return {"y": sample(np.concatenate(want))}


def _runs() -> dict:
    from tests import test_reference_build as t

    runs = {}
    for name in t.MODELS:
        for fast in (False, True):
            runs[f"wav/{name}/{regime(fast)}"] = functools.partial(
                _stream, fx.load_model(name), fx.input_wav()[43000:53000], fast)
    runs["wav_45000/wavenet_a1_standard/exact"] = functools.partial(
        _stream, fx.load_model("wavenet_a1_standard"), fx.input_wav()[45000:51000])
    for name in ("wavenet_a1_standard", "a2_full", "lstm"):
        for block in (64, 1000):
            runs[f"blocks/{name}/{block}"] = functools.partial(
                _stream, fx.load_model(name), fx.synthetic_batch(1, 3000, seed=17)[0], block=block)
    for name in ("wavenet", "wavenet_a1_standard", "a2_full"):
        runs[f"full_input/{name}"] = functools.partial(_full_input_decimated, name)
    for name in ("a2_lite", "a2_full"):
        for variant in ("default", "generic"):
            runs[f"a2_variants/{name}/{variant}"] = functools.partial(
                _stream, fx.load_model(name), fx.synthetic_batch(1, 4000, seed=3)[0], variant=variant)
    runs["container_semantics"] = _container_semantics
    cont = fx.make_container([(0.5, fx.load_model("a2_lite")), (1.0, fx.load_model("a2_full"))])
    for slim in (None, 0.3):
        runs[f"container/{slim}"] = functools.partial(_stream, cont, fx.synthetic_batch(1, 3000, seed=31)[0], slim=slim)
    for i, (_, nam) in enumerate(t._multichannel_models()):
        runs[f"multichannel/{i}"] = functools.partial(_planar, nam, False, 640, 64, 17)
    for i, kw in enumerate(t.CONVNETS):
        for fast in (False, True):
            runs[f"convnet/{i}/{regime(fast)}"] = functools.partial(_planar, t._convnet(**kw), fast, 960, 96, 23)
    for case in (0, 1):
        runs[f"slimmable/{case}"] = functools.partial(_slimmable, case)
    for impl in ("direct", "fft", "auto"):
        runs[f"linear/{impl}"] = functools.partial(_stream, t.linear_fir(impl), fx.synthetic_batch(1, 3000, seed=5)[0])
    for name in ("lstm", "wavenet"):
        runs[f"reset_prewarm/{name}"] = functools.partial(_reset_and_prewarm, name)
    return runs


def record() -> dict:
    """Every run on the reference build: {"<key>/<array>": array}."""
    return {f"{key}/{k}": v for key, run in _runs().items() for k, v in run().items()}


def main() -> None:
    from oracle import ref

    if not (ref.available() and ref.available("generic")):
        raise SystemExit("oracle/_ref/ is not built: run build() where the reference checkout is readable (NAM_REFERENCE)")
    arrays = record()
    np.savez_compressed(GOLDEN, **arrays)
    print(f"wrote {GOLDEN.name}: {len(arrays)} arrays, {GOLDEN.stat().st_size} bytes")


if __name__ == "__main__":
    main()
