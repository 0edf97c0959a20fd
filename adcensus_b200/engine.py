"""ctypes binding of the C ABI (include/adcensus_b200.h) and the Python mirror of the reference's
ADCensusStereo class.  Every call goes through libadcensus_b200.so; nothing is computed in Python."""
from __future__ import annotations

import ctypes
from pathlib import Path

import numpy as np

Invalid_Float = float("inf")  # reference adcensus_types.h:33

STAGES = ["COST", "ARMS", "AGG1", "AGG2", "AGG3", "AGG4", "SO1", "SO2", "SO3", "SO4",
          "WTA", "OUTLIER", "VOTE", "INTERP", "DISC", "MEDIAN"]
STAGE = {n: i for i, n in enumerate(STAGES)}
TAPS = ["GRAY_L", "GRAY_R", "CENSUS_L", "CENSUS_R", "VOL_INIT", "VOL_AGGR", "ARMS", "SUPCNT_H",
        "SUPCNT_V", "DISP_L", "DISP_R", "MISMATCHES", "OCCLUSIONS"]
TAP = {n: i for i, n in enumerate(TAPS)}
_TAP_DTYPE = {"GRAY_L": np.uint8, "GRAY_R": np.uint8, "CENSUS_L": np.uint64, "CENSUS_R": np.uint64,
              "VOL_INIT": np.float32, "VOL_AGGR": np.float32, "ARMS": np.uint8, "SUPCNT_H": np.uint16,
              "SUPCNT_V": np.uint16, "DISP_L": np.float32, "DISP_R": np.float32,
              "MISMATCHES": np.int32, "OCCLUSIONS": np.int32}


class ADCensusOption(ctypes.Structure):
    """Mirror of the reference's ADCensusOption (adcensus_types.h:45-75): same fields, order,
    types and defaults; 60 bytes, passed to the C ABI as-is."""
    _fields_ = [("min_disparity", ctypes.c_int32), ("max_disparity", ctypes.c_int32),
                ("lambda_ad", ctypes.c_int32), ("lambda_census", ctypes.c_int32),
                ("cross_L1", ctypes.c_int32), ("cross_L2", ctypes.c_int32),
                ("cross_t1", ctypes.c_int32), ("cross_t2", ctypes.c_int32),
                ("so_p1", ctypes.c_float), ("so_p2", ctypes.c_float),
                ("so_tso", ctypes.c_int32), ("irv_ts", ctypes.c_int32),
                ("irv_th", ctypes.c_float), ("lrcheck_thres", ctypes.c_float),
                ("do_lr_check", ctypes.c_bool), ("do_filling", ctypes.c_bool),
                ("do_discontinuity_adjustment", ctypes.c_bool), ("_reserved", ctypes.c_uint8)]

    def __init__(self, **kw):
        super().__init__(0, 64, 10, 30, 34, 17, 20, 6, 1.0, 3.0, 15, 20, 0.4, 1.0, True, True, False, 0)
        for k, v in kw.items():
            if k not in dict(self._fields_):
                raise AttributeError(f"ADCensusOption has no field {k!r}")
            setattr(self, k, v)


assert ctypes.sizeof(ADCensusOption) == 60


class _Config(ctypes.Structure):
    _fields_ = [("device", ctypes.c_int32), ("wave_pairs", ctypes.c_int32), ("lanes", ctypes.c_int32),
                ("debug_flags", ctypes.c_int32), ("max_disparity_range", ctypes.c_int32), ("reserved", ctypes.c_int32 * 11)]


assert ctypes.sizeof(_Config) == 64 and _Config.max_disparity_range.offset == 16

# adc_config.max_disparity_range: 0 = MAX_DISPARITY_RANGE; an engine may raise its limit up to MAX_DISPARITY_RANGE_WIDE
MAX_DISPARITY_RANGE, MAX_DISPARITY_RANGE_WIDE = 256, 512


# adc_config.debug_flags (test hooks)
DBG_NO_RAY_TABLE, DBG_VOTE_ENUM, DBG_VOTE_GLOBAL_STATE, DBG_UNFUSED_AGG = 1, 2, 4, 8


class AuxOutputs(ctypes.Structure):
    """Mirror of adc_aux_outputs: device or host pointers of the side outputs, 0 / None = not wanted."""
    _fields_ = [("origin", ctypes.c_void_p), ("cost_best", ctypes.c_void_p), ("cost_second", ctypes.c_void_p),
                ("disp_right", ctypes.c_void_p)]


assert ctypes.sizeof(AuxOutputs) == 32

# adc_aux_outputs.origin: how a pixel's value was obtained (before discontinuity adjustment and the median filter)
ADC_ORIGIN_MATCHED, ADC_ORIGIN_VOTED_MISMATCH, ADC_ORIGIN_VOTED_OCCLUSION = 0, 1, 2
ADC_ORIGIN_INTERP_MISMATCH, ADC_ORIGIN_INTERP_OCCLUSION, ADC_ORIGIN_INVALID = 3, 4, 5
ADC_ORIGIN_WTA_INVALID = 8   # flag OR-ed onto the code: WTA itself returned Invalid_Float
AUX_NAMES = ("origin", "cost_best", "cost_second", "disp_right")
_AUX_DTYPE = {"origin": np.uint8, "cost_best": np.float32, "cost_second": np.float32, "disp_right": np.float32}


class AdcError(RuntimeError):
    pass


def lib_path() -> Path:
    return Path(__file__).resolve().parent / "lib" / "libadcensus_b200.so"


_lib = None


def load_library() -> ctypes.CDLL:
    """Loads libadcensus_b200.so.  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not p.exists():
        raise AdcError(f"{p} is missing: build it with adcensus_b200.build_library() "
                       "(nvcc, sm_100a).  This package has no CPU fallback.")
    L = ctypes.CDLL(str(p))
    vp, i32, u8p, f32p = ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p
    L.adc_default_option.argtypes = [ctypes.POINTER(ADCensusOption)]
    L.adc_create.argtypes = [i32, i32, ctypes.POINTER(ADCensusOption), ctypes.POINTER(_Config), ctypes.POINTER(vp)]
    L.adc_create.restype = ctypes.c_int
    L.adc_destroy.argtypes = [vp]
    L.adc_destroy.restype = None
    L.adc_match.argtypes = [vp, u8p, u8p, f32p]
    L.adc_get_right_disparity.argtypes = [vp, f32p]
    L.adc_match_batch.argtypes = [vp, i32, ctypes.POINTER(vp), ctypes.POINTER(vp), ctypes.POINTER(vp)]
    L.adc_match_batch_strided.argtypes = [vp, i32, u8p, u8p, f32p]
    L.adc_match_batch_device.argtypes = [vp, i32, u8p, u8p, f32p, vp]
    L.adc_match_batch_pinned_async.argtypes = [vp, i32, u8p, u8p, f32p, vp]
    auxp = ctypes.POINTER(AuxOutputs)
    L.adc_match_aux.argtypes = [vp, u8p, u8p, f32p, auxp]
    L.adc_match_batch_strided_aux.argtypes = [vp, i32, u8p, u8p, f32p, auxp]
    L.adc_match_batch_device_aux.argtypes = [vp, i32, u8p, u8p, f32p, auxp, vp]
    L.adc_host_alloc.argtypes = [ctypes.c_size_t]
    L.adc_host_alloc.restype = vp
    L.adc_host_free.argtypes = [vp]
    L.adc_host_free.restype = None
    L.adc_synchronize.argtypes = [vp]
    L.adc_launch_count.argtypes = [vp]
    L.adc_launch_count.restype = ctypes.c_uint64
    L.adc_last_stage_ms.argtypes = [vp, ctypes.POINTER(ctypes.c_float * 6)]
    L.adc_get_config.argtypes = [vp, ctypes.POINTER(_Config)]
    L.adc_profile_kernel.argtypes = [vp, i32, i32, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_double)]
    L.adc_set_pipelined.argtypes = [vp, i32]
    L.adc_join.argtypes = [vp, vp]
    L.adc_render_disparity.argtypes = [vp, f32p, u8p, u8p, f32p]
    L.adc_disparity_cloud.argtypes = [vp, u8p, f32p, f32p, ctypes.POINTER(ctypes.c_int32)]
    L.adc_last_error.restype = ctypes.c_char_p
    L.adc_version.restype = ctypes.c_char_p
    L.adc_debug_run.argtypes = [vp, u8p, u8p, i32]
    L.adc_debug_get.argtypes = [vp, i32, vp, ctypes.c_size_t]
    L.adc_debug_get.restype = ctypes.c_size_t
    L.adc_debug_counters.argtypes = [vp, ctypes.POINTER(ctypes.c_int32 * 16)]
    _lib = L
    return L


def _check(rc: int):
    if rc != 0:
        raise AdcError(f"adcensus_b200 error {rc}: {load_library().adc_last_error().decode()}")


def _img(a, shape) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if a.shape != shape:
        raise ValueError(f"expected packed BGR uint8 array of shape {shape}, got {a.shape}")
    return a


class Engine:
    """Thin object wrapper over adc_create/.../adc_destroy."""

    def __init__(self, width: int, height: int, option: ADCensusOption | None = None, device: int = 0,
                 wave_pairs: int = 0, lanes: int = 0, debug_flags: int = 0, max_disparity_range: int = 0):
        """max_disparity_range: the largest max_disparity - min_disparity this engine accepts; 0 = MAX_DISPARITY_RANGE,
        at most MAX_DISPARITY_RANGE_WIDE."""
        self._L = load_library()
        self.width, self.height = int(width), int(height)
        self.option = option or ADCensusOption()
        self.D = self.option.max_disparity - self.option.min_disparity
        cfg = _Config(device=device, wave_pairs=wave_pairs, lanes=lanes, debug_flags=debug_flags,
                      max_disparity_range=max_disparity_range)
        h = ctypes.c_void_p()
        _check(self._L.adc_create(self.width, self.height, ctypes.byref(self.option), ctypes.byref(cfg), ctypes.byref(h)))
        self._h = h
        got = _Config()
        self._L.adc_get_config(self._h, ctypes.byref(got))
        self.wave_pairs, self.lanes, self.device = got.wave_pairs, got.lanes, got.device
        self.max_disparity_range = got.max_disparity_range

    def close(self):
        if getattr(self, "_h", None):
            self._L.adc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- Match ----------------------------------------------------------------------------
    def match(self, left, right) -> np.ndarray:
        left = _img(left, (self.height, self.width, 3))
        right = _img(right, (self.height, self.width, 3))
        disp = np.empty((self.height, self.width), np.float32)
        _check(self._L.adc_match(self._h, left.ctypes.data, right.ctypes.data, disp.ctypes.data))
        return disp

    def right_disparity(self) -> np.ndarray:
        """Right-view map of the most recent match() (the reference's private disp_right_)."""
        disp = np.empty((self.height, self.width), np.float32)
        _check(self._L.adc_get_right_disparity(self._h, disp.ctypes.data))
        return disp

    def match_batch(self, lefts, rights) -> np.ndarray:
        """lefts/rights: arrays [n][H][W][3] (or sequences of images).  Host memory in, host memory out."""
        lefts = np.ascontiguousarray(lefts, np.uint8)
        rights = np.ascontiguousarray(rights, np.uint8)
        n = lefts.shape[0]
        if lefts.shape != (n, self.height, self.width, 3) or rights.shape != lefts.shape:
            raise ValueError("expected [n][H][W][3] uint8 arrays")
        disp = np.empty((n, self.height, self.width), np.float32)
        _check(self._L.adc_match_batch_strided(self._h, n, lefts.ctypes.data, rights.ctypes.data, disp.ctypes.data))
        return disp

    def _aux_arrays(self, want, lead=()):
        unknown = set(want) - set(AUX_NAMES)
        if unknown:
            raise ValueError(f"unknown side outputs {sorted(unknown)}; choose from {AUX_NAMES}")
        out = {k: np.empty(lead + (self.height, self.width), _AUX_DTYPE[k]) for k in AUX_NAMES if k in want}
        return out, AuxOutputs(**{k: a.ctypes.data for k, a in out.items()})

    def match_aux(self, left, right, want=AUX_NAMES):
        """match() with side outputs: (disp, {name: [H][W] array}) for the names in `want` (AUX_NAMES)."""
        left = _img(left, (self.height, self.width, 3))
        right = _img(right, (self.height, self.width, 3))
        disp = np.empty((self.height, self.width), np.float32)
        out, aux = self._aux_arrays(want)
        _check(self._L.adc_match_aux(self._h, left.ctypes.data, right.ctypes.data, disp.ctypes.data, ctypes.byref(aux)))
        return disp, out

    def match_batch_aux(self, lefts, rights, want=AUX_NAMES):
        """match_batch() with side outputs: (disp [n][H][W], {name: [n][H][W] array})."""
        lefts = np.ascontiguousarray(lefts, np.uint8)
        rights = np.ascontiguousarray(rights, np.uint8)
        n = lefts.shape[0]
        if lefts.shape != (n, self.height, self.width, 3) or rights.shape != lefts.shape:
            raise ValueError("expected [n][H][W][3] uint8 arrays")
        disp = np.empty((n, self.height, self.width), np.float32)
        out, aux = self._aux_arrays(want, (n,))
        _check(self._L.adc_match_batch_strided_aux(self._h, n, lefts.ctypes.data, rights.ctypes.data, disp.ctypes.data,
                                                   ctypes.byref(aux)))
        return disp, out

    def match_batch_device_aux(self, n: int, d_left: int, d_right: int, d_disp: int, origin: int = 0, cost_best: int = 0,
                               cost_second: int = 0, disp_right: int = 0, stream: int = 0):
        """match_batch_device() with side outputs into device buffers (ints, 0 = not wanted), [n][H][W] each."""
        aux = AuxOutputs(origin or None, cost_best or None, cost_second or None, disp_right or None)
        _check(self._L.adc_match_batch_device_aux(self._h, n, d_left, d_right, d_disp, ctypes.byref(aux), stream))

    def match_batch_ptrs(self, lefts, rights):
        """Pointer-array form (adc_match_batch): independent per-pair buffers."""
        n = len(lefts)
        ls = [_img(a, (self.height, self.width, 3)) for a in lefts]
        rs = [_img(a, (self.height, self.width, 3)) for a in rights]
        ds = [np.empty((self.height, self.width), np.float32) for _ in range(n)]
        arr = ctypes.c_void_p * n
        _check(self._L.adc_match_batch(self._h, n, arr(*[a.ctypes.data for a in ls]),
                                       arr(*[a.ctypes.data for a in rs]), arr(*[a.ctypes.data for a in ds])))
        return ds

    def match_batch_device(self, n: int, d_left: int, d_right: int, d_disp: int, stream: int = 0):
        """Device pointers (ints), enqueued on `stream` (cudaStream_t as int) without synchronising."""
        _check(self._L.adc_match_batch_device(self._h, n, d_left, d_right, d_disp, stream))

    def match_batch_pinned_async(self, n: int, left_ptr: int, right_ptr: int, disp_ptr: int, stream: int = 0):
        _check(self._L.adc_match_batch_pinned_async(self._h, n, left_ptr, right_ptr, disp_ptr, stream))

    def synchronize(self):
        _check(self._L.adc_synchronize(self._h))

    @property
    def launch_count(self) -> int:
        return int(self._L.adc_launch_count(self._h))

    def last_stage_ms(self):
        out = (ctypes.c_float * 6)()
        _check(self._L.adc_last_stage_ms(self._h, ctypes.byref(out)))
        return list(out)

    PROFILE_KERNELS = {"cost_volume": 0, "arm_sum_h": 1, "arm_sum_v_div": 2, "scanline_x": 3, "scanline_y": 4, "wta": 5,
                       "arm_sum2_v": 6, "arm_sum2_h": 7, "arm_sum_h_div": 8, "arm_sum_v": 9, "wta_aux": 10}

    def profile_kernel(self, name: str, reps: int = 5):
        """(mean ms per launch over one wave, algorithmic bytes per launch) of one pipeline kernel."""
        ms, by = ctypes.c_float(), ctypes.c_double()
        _check(self._L.adc_profile_kernel(self._h, self.PROFILE_KERNELS[name], reps, ctypes.byref(ms), ctypes.byref(by)))
        return ms.value, by.value

    # ---- streaming: consecutive async batch calls without a drain in between -------------------
    def set_pipelined(self, on: bool = True):
        _check(self._L.adc_set_pipelined(self._h, 1 if on else 0))

    def join(self, stream: int = 0):
        """Makes `stream` wait for everything submitted so far (required before results are read in pipelined mode)."""
        _check(self._L.adc_join(self._h, stream))

    # ---- output side of the reference's demo (main.cpp:147-230) -------------------------------
    def render_disparity(self, disp: np.ndarray):
        """(gray8 [H][W], jet_bgr [H][W][3], (min, max)): SaveDisparityMap's two images (main.cpp:180-207)."""
        disp = np.ascontiguousarray(disp, np.float32).reshape(self.height, self.width)
        gray = np.empty((self.height, self.width), np.uint8)
        jet = np.empty((self.height, self.width, 3), np.uint8)
        mm = np.empty(2, np.float32)
        _check(self._L.adc_render_disparity(self._h, disp.ctypes.data, gray.ctypes.data, jet.ctypes.data, mm.ctypes.data))
        return gray, jet, (float(mm[0]), float(mm[1]))

    def disparity_cloud(self, left: np.ndarray, disp: np.ndarray) -> np.ndarray:
        """[n][6] float32 records (x, y, |d|, r, g, b) of the valid pixels in raster order (main.cpp:209-230)."""
        left = _img(left, (self.height, self.width, 3))
        disp = np.ascontiguousarray(disp, np.float32).reshape(self.height, self.width)
        cloud = np.empty((self.height * self.width, 6), np.float32)
        n = ctypes.c_int32(0)
        _check(self._L.adc_disparity_cloud(self._h, left.ctypes.data, disp.ctypes.data, cloud.ctypes.data, ctypes.byref(n)))
        return cloud[:n.value].copy()

    # ---- debug taps -------------------------------------------------------------------------
    def debug_run(self, left, right, last_stage: str):
        left = _img(left, (self.height, self.width, 3))
        right = _img(right, (self.height, self.width, 3))
        _check(self._L.adc_debug_run(self._h, left.ctypes.data, right.ctypes.data, STAGE[last_stage]))

    def counters(self):
        out = (ctypes.c_int32 * 16)()
        _check(self._L.adc_debug_counters(self._h, ctypes.byref(out)))
        return list(out)

    def tap(self, name: str) -> np.ndarray:
        tid = TAP[name]
        nbytes = self._L.adc_debug_get(self._h, tid, None, 0)
        buf = np.empty(nbytes, np.uint8)
        if nbytes:
            got = self._L.adc_debug_get(self._h, tid, buf.ctypes.data, nbytes)
            if got != nbytes:
                raise AdcError(f"adc_debug_get({name}) failed: {self._L.adc_last_error().decode()}")
        a = buf.view(_TAP_DTYPE[name])
        if name in ("VOL_INIT", "VOL_AGGR"):
            return a.reshape(self.height, self.width, self.D)
        if name == "ARMS":
            return a.reshape(self.height, self.width, 4)
        if name in ("MISMATCHES", "OCCLUSIONS"):
            return a.reshape(-1, 2)
        return a.reshape(self.height, self.width)


class ADCensusStereo:
    """Python mirror of the reference class (ADCensusStereo.h:14-95): Initialize / Match / Reset
    with the reference's bool-returning error behaviour."""

    def __init__(self):
        self._engine = None
        self._max_disparity_range = 0
        self.last_error = ""

    def Initialize(self, width: int, height: int, option: ADCensusOption, max_disparity_range: int = 0) -> bool:
        """max_disparity_range (extension, not in the reference): the engine's disparity range limit, see Engine."""
        self.Release()
        self._max_disparity_range = max_disparity_range
        try:
            self._engine = Engine(width, height, option, max_disparity_range=max_disparity_range)
        except (AdcError, ValueError) as e:
            self.last_error = str(e)
            self._engine = None
            return False
        return True

    def Match(self, img_left, img_right, disp_left: np.ndarray | None = None):
        """Returns False (like the reference) when not initialised or when an image is None;
        otherwise fills/returns the float32 disparity map."""
        if self._engine is None or img_left is None or img_right is None:
            return False
        out = self._engine.match(img_left, img_right)
        if disp_left is not None:
            np.copyto(disp_left.reshape(out.shape), out)
            return True
        return out

    def MatchWithConfidence(self, img_left, img_right):
        """Extension (not in the reference): (disp, origin, cost_best, cost_second) of one pair, see Engine.match_aux;
        False where Match returns False."""
        if self._engine is None or img_left is None or img_right is None:
            return False
        disp, aux = self._engine.match_aux(img_left, img_right, ("origin", "cost_best", "cost_second"))
        return disp, aux["origin"], aux["cost_best"], aux["cost_second"]

    def Reset(self, width: int, height: int, option: ADCensusOption) -> bool:
        self.Release()
        return self.Initialize(width, height, option, self._max_disparity_range)

    def Release(self):
        if self._engine is not None:
            self._engine.close()
        self._engine = None
