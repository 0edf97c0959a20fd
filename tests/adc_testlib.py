"""Shared helpers for the test-suite, tools/ and bench.py's CPU-baseline legs.

TEST INFRASTRUCTURE: this module is the only Python entry to the CPU checkers under ``oracle/``
(``oracle/_build/libadc_oracle.so`` = our C restatement, ``oracle/_ref/libadcensus_ref.so`` = the
unmodified reference behind a harness).  The product package ``adcensus_b200`` never imports it.
"""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent.parent
ORACLE_DIR = REPO / "oracle"
GOLDEN_DIR = REPO / "tests" / "golden"
REFERENCE_ROOT = Path("/root/reference")

# stage / tap ids (oracle/adc_taps.h == include/adcensus_b200.h)
STAGES = ["COST", "ARMS", "AGG1", "AGG2", "AGG3", "AGG4", "SO1", "SO2", "SO3", "SO4",
          "WTA", "OUTLIER", "VOTE", "INTERP", "DISC", "MEDIAN"]
STAGE = {n: i for i, n in enumerate(STAGES)}
TAPS = ["GRAY_L", "GRAY_R", "CENSUS_L", "CENSUS_R", "VOL_INIT", "VOL_AGGR", "ARMS", "SUPCNT_H",
        "SUPCNT_V", "DISP_L", "DISP_R", "MISMATCHES", "OCCLUSIONS"]
TAP = {n: i for i, n in enumerate(TAPS)}
TAP_DTYPE = {"GRAY_L": np.uint8, "GRAY_R": np.uint8, "CENSUS_L": np.uint64, "CENSUS_R": np.uint64,
             "VOL_INIT": np.float32, "VOL_AGGR": np.float32, "ARMS": np.uint8, "SUPCNT_H": np.uint16,
             "SUPCNT_V": np.uint16, "DISP_L": np.float32, "DISP_R": np.float32,
             "MISMATCHES": np.int32, "OCCLUSIONS": np.int32}
# which buffers are meaningful right after a stage (what the parity tests compare)
STAGE_TAPS = {
    "COST": ["GRAY_L", "GRAY_R", "CENSUS_L", "CENSUS_R", "VOL_INIT"],
    "ARMS": ["ARMS", "SUPCNT_H", "SUPCNT_V"],
    "AGG1": ["VOL_AGGR"], "AGG2": ["VOL_AGGR"], "AGG3": ["VOL_AGGR"], "AGG4": ["VOL_AGGR"],
    "SO1": ["VOL_INIT"], "SO2": ["VOL_AGGR"], "SO3": ["VOL_INIT"], "SO4": ["VOL_AGGR"],
    "WTA": ["DISP_L", "DISP_R"],
    "OUTLIER": ["DISP_L", "MISMATCHES", "OCCLUSIONS"],
    "VOTE": ["DISP_L", "MISMATCHES", "OCCLUSIONS"],
    "INTERP": ["DISP_L"], "DISC": ["DISP_L"], "MEDIAN": ["DISP_L"],
}


class Option(ctypes.Structure):
    """Byte-identical to the reference's ADCensusOption (adcensus_types.h:45-75), 60 bytes."""
    _fields_ = [("min_disparity", ctypes.c_int32), ("max_disparity", ctypes.c_int32),
                ("lambda_ad", ctypes.c_int32), ("lambda_census", ctypes.c_int32),
                ("cross_L1", ctypes.c_int32), ("cross_L2", ctypes.c_int32),
                ("cross_t1", ctypes.c_int32), ("cross_t2", ctypes.c_int32),
                ("so_p1", ctypes.c_float), ("so_p2", ctypes.c_float),
                ("so_tso", ctypes.c_int32), ("irv_ts", ctypes.c_int32),
                ("irv_th", ctypes.c_float), ("lrcheck_thres", ctypes.c_float),
                ("do_lr_check", ctypes.c_uint8), ("do_filling", ctypes.c_uint8),
                ("do_discontinuity_adjustment", ctypes.c_uint8), ("_pad", ctypes.c_uint8)]


def default_option(**kw) -> Option:
    o = Option(0, 64, 10, 30, 34, 17, 20, 6, 1.0, 3.0, 15, 20, 0.4, 1.0, 1, 1, 0, 0)
    for k, v in kw.items():
        setattr(o, k, v)
    return o


assert ctypes.sizeof(Option) == 60


# ------------------------------------------------------------------------------------------------
def build_oracle(force: bool = False) -> None:
    """Compile the C restatement (always) and the reference harness (when /root/reference exists)."""
    target = ORACLE_DIR / "_build" / "libadc_oracle.so"
    srcs = [ORACLE_DIR / f for f in ("adc_oracle.c", "adc_oracle.h", "adc_taps.h")]
    if force or not target.exists() or any(s.stat().st_mtime > target.stat().st_mtime for s in srcs):
        subprocess.run(["make", "-C", str(ORACLE_DIR), "oracle"], check=True, capture_output=True)
    ref = ORACLE_DIR / "_ref" / "libadcensus_ref.so"
    # os.access, not Path.is_dir: a user who may not enter the reference's parent directory gets
    # False here instead of a PermissionError, and keeps the committed goldens as the only pin
    if os.access(REFERENCE_ROOT / "AD-Census", os.R_OK | os.X_OK):
        if force or not ref.exists() or (ORACLE_DIR / "ref_harness.cpp").stat().st_mtime > ref.stat().st_mtime:
            subprocess.run(["make", "-C", str(ORACLE_DIR), "ref"], check=True, capture_output=True)


def have_ref() -> bool:
    return (ORACLE_DIR / "_ref" / "libadcensus_ref.so").exists()


class _Checker:
    """Common ctypes wrapper: both CPU checkers export the same staged API under two prefixes."""

    def __init__(self, libpath: Path, prefix: str, width: int, height: int, opt: Option):
        self.lib = ctypes.CDLL(str(libpath))
        self.p = prefix
        f = self._f
        f("create").restype = ctypes.c_void_p
        f("create").argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        f("destroy").argtypes = [ctypes.c_void_p]
        f("begin").argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        f("step").argtypes = [ctypes.c_void_p]
        f("tap").restype = ctypes.c_size_t
        f("tap").argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t]
        f("time_match").restype = ctypes.c_double
        f("time_match").argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        self.w, self.h = width, height
        self.opt = opt
        self.D = opt.max_disparity - opt.min_disparity
        self.ctx = f("create")(width, height, ctypes.byref(opt))
        self._keep = None

    def _f(self, name):
        return getattr(self.lib, f"{self.p}_{name}")

    @property
    def ok(self) -> bool:
        return bool(self.ctx)

    def close(self):
        if self.ctx:
            self._f("destroy")(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def begin(self, left: np.ndarray, right: np.ndarray):
        left = np.ascontiguousarray(left, np.uint8)
        right = np.ascontiguousarray(right, np.uint8)
        self._keep = (left, right)
        assert self._f("begin")(self.ctx, left.ctypes.data, right.ctypes.data) == 1

    def step(self) -> int:
        return self._f("step")(self.ctx)

    def run_to(self, stage: str):
        """Run stages until `stage` (inclusive) has executed."""
        target = STAGE[stage]
        while True:
            s = self.step()
            if s < 0 or s >= target:
                return

    def tap(self, name: str) -> np.ndarray:
        tid = TAP[name]
        nbytes = self._f("tap")(self.ctx, tid, None, 0)
        buf = np.empty(nbytes, np.uint8)
        if nbytes:
            self._f("tap")(self.ctx, tid, buf.ctypes.data, nbytes)
        a = buf.view(TAP_DTYPE[name])
        n = self.w * self.h
        if name in ("VOL_INIT", "VOL_AGGR"):
            return a.reshape(self.h, self.w, self.D)
        if name == "ARMS":
            return a.reshape(self.h, self.w, 4)
        if name in ("MISMATCHES", "OCCLUSIONS"):
            return a.reshape(-1, 2)
        return a.reshape(self.h, self.w) if a.size == n else a

    def match(self, left: np.ndarray, right: np.ndarray) -> np.ndarray:
        self.begin(left, right)
        while self.step() >= 0:
            pass
        return self.tap("DISP_L").copy()

    def time_match(self, left, right, iters=1) -> float:
        left = np.ascontiguousarray(left, np.uint8)
        right = np.ascontiguousarray(right, np.uint8)
        disp = np.empty((self.h, self.w), np.float32)
        return self._f("time_match")(self.ctx, left.ctypes.data, right.ctypes.data, disp.ctypes.data, iters)


class Oracle(_Checker):
    """Our C restatement (oracle/adc_oracle.c)."""

    def __init__(self, width, height, opt=None):
        build_oracle()
        super().__init__(ORACLE_DIR / "_build" / "libadc_oracle.so", "orc", width, height, opt or default_option())


class Reference(_Checker):
    """The unmodified reference (oracle/_ref), available where it was built."""

    def __init__(self, width, height, opt=None):
        super().__init__(ORACLE_DIR / "_ref" / "libadcensus_ref.so", "ref", width, height, opt or default_option())

    def stock_match(self, left, right) -> np.ndarray:
        """ADCensusStereo::Match itself (not the staged runner)."""
        self.lib.ref_match.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int]
        left = np.ascontiguousarray(left, np.uint8)
        right = np.ascontiguousarray(right, np.uint8)
        disp = np.empty((self.h, self.w), np.float32)
        assert self.lib.ref_match(self.ctx, left.ctypes.data, right.ctypes.data, disp.ctypes.data, 1) == 1
        return disp


# ------------------------------------------------------------------------------------------------
def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def load_cone():
    """The Cone pair (reference Data/Cone/im2.png = left, im6.png = right) as packed BGR u8,
    from the committed fixture (the GPU box has no /root/reference)."""
    z = np.load(GOLDEN_DIR / "cone_pair.npz")
    return z["left"], z["right"]


_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def _splitmix64(x: np.ndarray) -> np.ndarray:
    with np.errstate(over="ignore"):
        x = (x + np.uint64(0x9E3779B97F4A7C15)) & _M64
        z = x
        z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & _M64
        z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & _M64
        return z ^ (z >> np.uint64(31))


def synthetic_pair(width: int, height: int, disp_range: int, seed: int):
    """Deterministic textured stereo pair (SURVEY.md section 8d): three octaves of bilinearly
    interpolated hash lattices, right view = left view shifted by a per-25-row band disparity.
    NOT white noise on purpose: cross arms must have realistic lengths."""
    D = int(disp_range)
    Wt = width + 2 * D
    tex = np.zeros((height, Wt, 3), np.float64)
    ys = np.arange(height)[:, None]
    xs = np.arange(Wt)[None, :]
    with np.errstate(over="ignore"):
        for o, (period, weight) in enumerate(((64, 0.55), (16, 0.30), (4, 0.15))):
            j0, fy = ys // period, (ys % period) / period
            i0, fx = xs // period, (xs % period) / period
            for c in range(3):
                def lat(j, i):
                    key = (np.uint64(seed) ^ (np.uint64(o) * np.uint64(0xD6E8FEB86659FD93))
                           ^ (j.astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15))
                           ^ (i.astype(np.uint64) * np.uint64(0xC2B2AE3D27D4EB4F))
                           ^ (np.uint64(c) * np.uint64(0x165667B19E3779F9)))
                    return (_splitmix64(key) & np.uint64(0xFF)).astype(np.float64)
                v = (lat(j0, i0) * (1 - fy) * (1 - fx) + lat(j0, i0 + 1) * (1 - fy) * fx
                     + lat(j0 + 1, i0) * fy * (1 - fx) + lat(j0 + 1, i0 + 1) * fy * fx)
                tex[:, :, c] += weight * v
    tex = np.floor(tex + 0.5).clip(0, 255).astype(np.uint8)
    left = np.ascontiguousarray(tex[:, D:D + width])
    right = np.empty_like(left)
    lo = D // 8
    span = max(1, (3 * D) // 4 - lo)
    with np.errstate(over="ignore"):
        bands = _splitmix64(np.uint64(seed) * np.uint64(1000003) + (np.arange(height) // 25).astype(np.uint64))
    for y in range(height):
        db = lo + int(bands[y] % np.uint64(span))
        right[y] = tex[y, D + db:D + db + width]
    return left, right


def crop_pair(left, right, x0, y0, w, h):
    return (np.ascontiguousarray(left[y0:y0 + h, x0:x0 + w]), np.ascontiguousarray(right[y0:y0 + h, x0:x0 + w]))
