"""ctypes front-end for oracle/_ref/libnam_ref.so: the UNMODIFIED reference (NeuralAmpModelerCore) compiled from
its own sources against oracle/eigen_shim (recipe: `make -C oracle ref`, run by build() where the reference checkout
-- oracle/Makefile's REF, or the NAM_REFERENCE environment variable -- is readable; the .so is git-ignored).

TEST INFRASTRUCTURE ONLY, like the rest of oracle/: it pins the C restatement (nam_oracle.c) and the CUDA path
against the reference's own code at whole-model level.  Nothing in the product imports this module.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
REF_DIR = HERE / "_ref"
_LIBS: dict[str, C.CDLL] = {}


def lib_path(variant: str = "default") -> Path:
    names = {"default": "libnam_ref.so", "generic": "libnam_ref_generic.so", "fast": "libnam_ref_fast.so",
             "fast512": "libnam_ref_fast512.so"}
    return REF_DIR / names[variant]


def available(variant: str = "default") -> bool:
    return lib_path(variant).exists()


def reference_tree() -> Path | None:
    """The reference checkout: NAM_REFERENCE if set, else oracle/Makefile's REF default; None where it is absent or not
    readable by this user."""
    tree = os.environ.get("NAM_REFERENCE") or subprocess.run(
        ["make", "-s", "--no-print-directory", "-C", str(HERE), "ref_tree"], capture_output=True, text=True,
        check=True).stdout.strip()
    try:
        return Path(tree) if (Path(tree) / "NAM" / "dsp.cpp").is_file() else None
    except OSError:  # a directory on the way this user may not enter
        return None


def build(force: bool = False) -> bool:
    """Compile the reference and its tools from reference_tree(); returns False (and builds nothing) without one."""
    tree = reference_tree()
    if tree is None:
        return False
    cmd = ["make", "-C", str(HERE), "ref", "ref_tools", f"REF={tree}"] + (["-B"] if force else [])
    subprocess.run(cmd, check=True, capture_output=True)
    return True


def _load(variant: str) -> C.CDLL:
    if variant not in _LIBS:
        lib = C.CDLL(str(lib_path(variant)))
        lib.namref_create.restype = C.c_void_p
        lib.namref_create.argtypes = [C.c_char_p, C.c_int]
        lib.namref_destroy.argtypes = [C.c_void_p]
        lib.namref_last_error.restype = C.c_char_p
        lib.namref_reset.argtypes = [C.c_void_p, C.c_double, C.c_int]
        lib.namref_process_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        lib.namref_run_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_long, C.c_int]
        lib.namref_process_planar_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        lib.namref_set_slimmable_size.argtypes = [C.c_void_p, C.c_double]
        if hasattr(lib, "namref_prewarm"):
            lib.namref_prewarm.argtypes = [C.c_void_p]
        for name in ("prewarm_samples", "in_channels", "out_channels"):
            getattr(lib, f"namref_{name}").argtypes = [C.c_void_p]
        lib.namref_expected_sample_rate.argtypes = [C.c_void_p]
        lib.namref_expected_sample_rate.restype = C.c_double
        _LIBS[variant] = lib
    return _LIBS[variant]


class ReferenceError_(RuntimeError):
    pass


class ReferenceModel:
    """nam::get_dsp(path) -> Reset -> process, through the reference's public API.

    NOTE the fast-tanh switch is process-global in the reference (NAM/activations.cpp:168-177): it is set at load
    time and read again by the LSTM at run time, so keep one regime alive at a time per process."""

    def __init__(self, path: str | os.PathLike, fast_tanh: bool = False, variant: str = "default"):
        self._lib = _load(variant)
        self._h = self._lib.namref_create(str(path).encode(), int(bool(fast_tanh)))
        if not self._h:
            raise ReferenceError_(self._lib.namref_last_error().decode(errors="replace"))

    @classmethod
    def from_dict(cls, nam: dict, fast_tanh: bool = False, variant: str = "default") -> "ReferenceModel":
        with tempfile.NamedTemporaryFile("w", suffix=".nam", delete=False) as f:
            json.dump(nam, f)
            path = f.name
        try:
            return cls(path, fast_tanh, variant)
        finally:
            os.unlink(path)

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.namref_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def prewarm_samples(self) -> int:
        return int(self._lib.namref_prewarm_samples(self._h))

    @property
    def expected_sample_rate(self) -> float:
        return float(self._lib.namref_expected_sample_rate(self._h))

    def reset(self, sample_rate: float, max_buffer_size: int) -> None:
        if self._lib.namref_reset(self._h, float(sample_rate), int(max_buffer_size)) != 0:
            raise ReferenceError_(self._lib.namref_last_error().decode(errors="replace"))

    def prewarm(self) -> None:
        """DSP::prewarm() from the current state."""
        if self._lib.namref_prewarm(self._h) != 0:
            raise ReferenceError_(self._lib.namref_last_error().decode(errors="replace"))

    def set_slimmable_size(self, value: float) -> None:
        if self._lib.namref_set_slimmable_size(self._h, float(value)) != 0:
            raise ReferenceError_(self._lib.namref_last_error().decode(errors="replace"))

    @property
    def in_channels(self) -> int:
        return int(self._lib.namref_in_channels(self._h))

    @property
    def out_channels(self) -> int:
        return int(self._lib.namref_out_channels(self._h))

    def process_planar(self, x: np.ndarray) -> np.ndarray:
        """One DSP::process call on x (in_channels, n) -> (out_channels, n); n <= the last reset's maxBufferSize."""
        x = np.ascontiguousarray(x, np.float32)
        assert x.ndim == 2 and x.shape[0] == self.in_channels
        y = np.zeros((self.out_channels, x.shape[1]), np.float32)
        if self._lib.namref_process_planar_f32(self._h, x.ctypes.data, y.ctypes.data, x.shape[1]) != 0:
            raise ReferenceError_(self._lib.namref_last_error().decode(errors="replace"))
        return y

    def run(self, x: np.ndarray, block: int) -> np.ndarray:
        """Mono signal through DSP::process in `block`-frame calls (block <= the last reset's maxBufferSize)."""
        x = np.ascontiguousarray(x, np.float32)
        y = np.zeros_like(x)
        if self._lib.namref_run_f32(self._h, x.ctypes.data, y.ctypes.data, len(x), int(block)) != 0:
            raise ReferenceError_(self._lib.namref_last_error().decode(errors="replace"))
        return y


def best_timed_variant() -> str | None:
    """The -Ofast build (tools/CMakeLists.txt:106) for the best ISA level this host has: "fast512" (x86-64-v4) or "fast"
    (x86-64-v3); None when neither was built."""
    try:
        flags = Path("/proc/cpuinfo").read_text()
    except OSError:
        flags = ""
    if all(f in flags for f in ("avx512f", "avx512bw", "avx512dq", "avx512vl")) and available("fast512"):
        return "fast512"
    if "avx2" in flags and "fma" in flags and available("fast"):
        return "fast"
    return None


class ReferencePool:
    """`streams` independent reference DSP objects (nam::get_dsp of the same file), each carrying its own state across
    process() calls, spread over host threads -- the reference's own code under the reference tools' protocol
    (tools/benchmodel.cpp:116-133: Reset(sr, 64), then 64-frame process() calls).  CPU-baseline timing only."""

    def __init__(self, nam: dict, streams: int, fast_tanh: bool, variant: str, block: int = 64):
        self.block = int(block)
        self.models = []
        with tempfile.NamedTemporaryFile("w", suffix=".nam", delete=False) as f:
            json.dump(nam, f)
            path = f.name
        try:
            for _ in range(int(streams)):
                m = ReferenceModel(path, fast_tanh, variant)
                m.reset(48000.0, self.block)
                self.models.append(m)
        finally:
            os.unlink(path)

    def process(self, x: np.ndarray, out: np.ndarray, threads: int) -> None:
        from concurrent.futures import ThreadPoolExecutor

        assert x.dtype == np.float32 and x.shape[0] == len(self.models) and x.flags["C_CONTIGUOUS"]
        lib = self.models[0]._lib
        n = x.shape[1]

        def work(t: int) -> None:  # ctypes releases the GIL for the duration of the foreign call
            for i in range(t, len(self.models), threads):
                if lib.namref_run_f32(self.models[i]._h, x[i].ctypes.data, out[i].ctypes.data, n, self.block) != 0:
                    raise ReferenceError_(lib.namref_last_error().decode(errors="replace"))

        with ThreadPoolExecutor(max_workers=threads) as ex:
            list(ex.map(work, range(threads)))

    def close(self) -> None:
        for m in self.models:
            m.close()
        self.models = []
