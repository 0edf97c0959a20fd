"""Per-pixel side outputs (adc_aux_outputs): origin, cost_best, cost_second and the right-view map, per pair.

CPU: the header and the ctypes mirror against the C struct's layout, the argument truth table of the three entry points
and of MatchWithConfidence, the oracle's side outputs against the unmodified reference's hashes
(tests/golden/golden_aux.json, written by tools/make_golden_aux.py), and what the outputs mean on Cone.
GPU: every golden case through adc_match_aux, the alternate voting paths, host and device batches over several waves and
two lanes (also pipelined), the launch count of the plain path, and the C++ class.
"""
import ctypes
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import adc_testlib as T

sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tools"))
import make_golden_aux as GA  # noqa: E402

CASE_IDS = [GA.case_key(c) for c in GA.AUX_CASES]
NAMES = ("origin", "cost_best", "cost_second", "disp_right")


def _golden():
    return json.loads(GA.JSON.read_text())


def _lib():
    import adcensus_b200 as A
    from adcensus_b200.build import build_library
    build_library()
    return A, A.load_library()


def _engine(w, h, opt, **kw):
    import adcensus_b200 as A
    o = A.ADCensusOption()
    for name, _ in T.Option._fields_:
        if not name.startswith("_"):
            setattr(o, name, getattr(opt, name))
    if opt.max_disparity - opt.min_disparity > 256:
        kw.setdefault("max_disparity_range", 512)
    return A.Engine(w, h, o, **kw)


def _same(name, got, want):
    assert got.shape == want.shape and got.dtype == want.dtype, f"{name}: {got.shape} {got.dtype} vs {want.shape} {want.dtype}"
    if not np.array_equal(got.view(np.uint8), want.view(np.uint8)):
        raise AssertionError(f"{name}: {int((got != want).sum())} of {got.size} values differ")


def _hashes(aux, disp, opt):
    return GA.aux_hashes(dict(aux, disp=disp), opt)


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_header_and_mirror_layout(tmp_path):
    """The header declares the struct, the three entry points and the origin codes; the library exports them; the ctypes
    mirror has the C struct's size and offsets (printed by a C program compiled against the header)."""
    A, L = _lib()
    hdr = (T.REPO / "include" / "adcensus_b200.h").read_text()
    assert "typedef struct adc_aux_outputs" in hdr
    for fn in ("adc_match_aux", "adc_match_batch_strided_aux", "adc_match_batch_device_aux"):
        assert f"int {fn}(" in hdr and hasattr(L, fn), fn
    codes = {"MATCHED": 0, "VOTED_MISMATCH": 1, "VOTED_OCCLUSION": 2, "INTERP_MISMATCH": 3, "INTERP_OCCLUSION": 4,
             "INVALID": 5, "WTA_INVALID": 8}
    from adcensus_b200 import engine as E
    for k, v in codes.items():
        assert f"ADC_ORIGIN_{k} = {v}" in hdr, k
        assert getattr(E, f"ADC_ORIGIN_{k}") == v, k
    probe = tmp_path / "probe.c"
    probe.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "adcensus_b200.h"\nint main(void) {\n'
                     '  printf("%zu %zu %zu %zu %zu\\n", sizeof(adc_aux_outputs), offsetof(adc_aux_outputs, origin),\n'
                     '         offsetof(adc_aux_outputs, cost_best), offsetof(adc_aux_outputs, cost_second),\n'
                     '         offsetof(adc_aux_outputs, disp_right));\n  return 0;\n}\n')
    r = subprocess.run(["gcc", str(probe), f"-I{T.REPO / 'include'}", "-o", str(tmp_path / "probe")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    c = [int(v) for v in subprocess.run([str(tmp_path / "probe")], capture_output=True, text=True).stdout.split()]
    py = [ctypes.sizeof(A.AuxOutputs)] + [getattr(A.AuxOutputs, n).offset for n in NAMES]
    assert c == py == [32, 0, 8, 16, 24]


def test_argument_errors_need_no_gpu():
    """ADC_ERR_ARG for a NULL engine, images or map and for n < 0, before any device work; Python's
    MatchWithConfidence returns False where Match does."""
    A, L = _lib()
    aux = A.AuxOutputs()
    img = np.zeros((4, 4, 3), np.uint8)
    disp = np.zeros((4, 4), np.float32)
    assert L.adc_match_aux(None, img.ctypes.data, img.ctypes.data, disp.ctypes.data, ctypes.byref(aux)) == 1
    assert L.adc_match_aux(None, None, None, None, None) == 1
    assert b"adc_match_aux" in L.adc_last_error()
    assert L.adc_match_batch_strided_aux(None, 1, img.ctypes.data, img.ctypes.data, disp.ctypes.data, ctypes.byref(aux)) == 1
    assert L.adc_match_batch_strided_aux(None, -1, None, None, None, None) == 1
    assert L.adc_match_batch_device_aux(None, 1, 1, 1, 1, ctypes.byref(aux), None) == 1
    assert L.adc_match_batch_device_aux(None, -1, None, None, None, None, None) == 1
    assert b"adc_match_batch_device_aux" in L.adc_last_error()
    s = A.ADCensusStereo()
    assert s.MatchWithConfidence(img, img) is False
    assert s.MatchWithConfidence(None, img) is False


@pytest.mark.parametrize("case", GA.AUX_CASES, ids=CASE_IDS)
def test_oracle_side_outputs_match_reference(case):
    """The side outputs derived from the oracle's stage taps hash to the ones derived from the unmodified reference."""
    g = _golden()[GA.case_key(case)]
    left, right, opt = GA.case_inputs(case)
    assert [T.sha(left), T.sha(right)] == g["input_sha"]
    h, w, _ = left.shape
    aux = GA.derive_aux(T.Oracle(w, h, opt), left, right, opt)
    assert GA.aux_hashes(aux, opt) == g["hashes"]


def _bad(disp, gt_u8):
    """Bad > 1 px per pixel on the known pixels of the Middlebury quarter-size ground truth (test_outputs.py's
    convention: value / 4, 0 = unknown, invalid = bad)."""
    known = gt_u8 > 0
    err = np.abs(np.where(np.isinf(disp), np.float32(1e9), disp) - gt_u8.astype(np.float32) / 4.0)
    return err > 1.0, known


def test_side_outputs_mean_what_they_say_on_cone():
    """On Cone: matched pixels are bad less often than filled ones, and among matched pixels the half with the lower
    cost_best / cost_second is bad less often than the other half."""
    left, right = T.load_cone()
    opt = T.default_option()
    aux = GA.derive_aux(T.Oracle(450, 375, opt), left, right, opt)
    gt = np.load(T.GOLDEN_DIR / "cone_gt.npz")["disp2"]
    bad, known = _bad(aux["disp"], gt)
    code = aux["origin"] & 7
    matched = known & (code == 0)
    filled = known & (code >= 1) & (code <= 4)
    assert matched.sum() > 0 and filled.sum() > 0
    assert bad[matched].mean() < bad[filled].mean()
    ratio = aux["cost_best"] / aux["cost_second"]
    med = np.median(ratio[matched])
    low, high = matched & (ratio <= med), matched & (ratio > med)
    assert bad[low].mean() < bad[high].mean()


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", GA.AUX_CASES, ids=CASE_IDS)
def test_match_aux_against_reference(case):
    """adc_match_aux: the four side outputs hash to the reference-derived values, and the map equals adc_match's."""
    g = _golden()[GA.case_key(case)]
    left, right, opt = GA.case_inputs(case)
    h, w, _ = left.shape
    eng = _engine(w, h, opt)
    disp, aux = eng.match_aux(left, right)
    assert _hashes(aux, disp, opt) == g["hashes"]
    _same("disp", disp, eng.match(left, right))
    _same("disp_right", aux["disp_right"], eng.right_disparity())
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("flag", ["DBG_VOTE_ENUM", "DBG_VOTE_GLOBAL_STATE"])
def test_origin_on_alternate_voting_paths(flag, cone):
    import adcensus_b200 as A
    left, right = cone
    g = _golden()["cone_full"]["hashes"]
    eng = _engine(450, 375, T.default_option(), debug_flags=getattr(A.engine, flag))
    disp, aux = eng.match_aux(left, right)
    assert _hashes(aux, disp, T.default_option()) == g
    eng.close()


def _batch_pairs(w, h, D, n, seed):
    pairs = [T.synthetic_pair(w, h, D, seed + i) for i in range(n)]
    return np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])


@pytest.mark.gpu
def test_batches_equal_single_pairs():
    """Host strided and device batches over three waves on two lanes, plain and pipelined: every pair's side outputs
    equal its single-pair adc_match_aux outputs, and disp_right equals adc_get_right_disparity after adc_match."""
    import torch
    w, h, D, n = 96, 40, 24, 5
    opt = T.default_option(max_disparity=D)
    lefts, rights = _batch_pairs(w, h, D, n, 300)
    eng = _engine(w, h, opt, wave_pairs=2, lanes=2)
    assert (eng.wave_pairs, eng.lanes) == (2, 2)
    single = []
    for i in range(n):
        d, aux = eng.match_aux(lefts[i], rights[i])
        _same(f"pair {i} disp", d, eng.match(lefts[i], rights[i]))
        _same(f"pair {i} disp_right", aux["disp_right"], eng.right_disparity())
        single.append((d, aux))
    disp, aux = eng.match_batch_aux(lefts, rights)
    for i, (d, a) in enumerate(single):
        _same(f"host pair {i} disp", disp[i], d)
        for k in NAMES:
            _same(f"host pair {i} {k}", aux[k][i], a[k])
    dev = torch.device("cuda", 0)
    dl, dr = torch.from_numpy(lefts).to(dev), torch.from_numpy(rights).to(dev)
    for pipelined in (False, True):
        eng.set_pipelined(pipelined)
        out = {"disp": torch.full((n, h, w), -1.0, device=dev), "origin": torch.full((n, h, w), 0xee, dtype=torch.uint8, device=dev),
               "cost_best": torch.full((n, h, w), -1.0, device=dev), "cost_second": torch.full((n, h, w), -1.0, device=dev),
               "disp_right": torch.full((n, h, w), -1.0, device=dev)}
        torch.cuda.synchronize()
        ptr = {k: v.data_ptr() for k, v in out.items()}
        img = h * w * 3
        for first, cnt in ((0, 3), (3, 2)):    # two calls: in pipelined mode the second flows into the first
            eng.match_batch_device_aux(cnt, dl.data_ptr() + first * img, dr.data_ptr() + first * img,
                                       ptr["disp"] + first * h * w * 4, origin=ptr["origin"] + first * h * w,
                                       cost_best=ptr["cost_best"] + first * h * w * 4,
                                       cost_second=ptr["cost_second"] + first * h * w * 4,
                                       disp_right=ptr["disp_right"] + first * h * w * 4)
        if pipelined:
            eng.join(0)
        torch.cuda.synchronize()
        got = {k: v.cpu().numpy() for k, v in out.items()}
        for i, (d, a) in enumerate(single):
            _same(f"device pair {i} disp (pipelined={pipelined})", got["disp"][i], d)
            for k in NAMES:
                _same(f"device pair {i} {k} (pipelined={pipelined})", got[k][i], a[k])
    eng.set_pipelined(False)
    eng.close()


@pytest.mark.gpu
def test_no_side_outputs_is_the_plain_path():
    """aux = NULL and an all-NULL struct issue exactly the plain call's launches and give its bits; disp_right alone adds
    no launch; all four add the origin kernel only (WTA runs as its side-output instantiation instead)."""
    import adcensus_b200 as A
    w, h, D = 96, 40, 24
    left, right = T.synthetic_pair(w, h, D, 77)
    eng = _engine(w, h, T.default_option(max_disparity=D))
    L = A.load_library()
    disp = np.empty((h, w), np.float32)

    def launches(fn):
        c0 = eng.launch_count
        out = fn()
        return eng.launch_count - c0, out

    n_plain, want = launches(lambda: eng.match(left, right))
    for aux in (None, ctypes.byref(A.AuxOutputs())):
        n, _ = launches(lambda: L.adc_match_aux(eng._h, left.ctypes.data, right.ctypes.data, disp.ctypes.data, aux))
        assert n == n_plain
        _same("disp", disp, want)
    n, (d, a) = launches(lambda: eng.match_aux(left, right, ("disp_right",)))
    assert n == n_plain and list(a) == ["disp_right"]
    _same("disp", d, want)
    n, _ = launches(lambda: eng.match_aux(left, right))
    assert n == n_plain + 1
    n_plain_b, want_b = launches(lambda: eng.match_batch(np.stack([left] * 3), np.stack([right] * 3)))
    n, (db, _) = launches(lambda: eng.match_batch_aux(np.stack([left] * 3), np.stack([right] * 3), ()))
    assert n == n_plain_b
    _same("batch disp", db, want_b)
    eng.close()


@pytest.mark.gpu
def test_cpp_match_with_confidence(tmp_path):
    """tests/cpp/confidence_main.cpp: MatchWithConfidence through the C++ class; its four buffers against the oracle."""
    import adcensus_b200 as A
    exe = tmp_path / "confidence"
    r = subprocess.run(["g++", "-std=c++17", str(T.REPO / "tests" / "cpp" / "confidence_main.cpp"), f"-I{T.REPO / 'include'}",
                        f"-L{A.lib_path().parent}", "-ladcensus_b200", f"-Wl,-rpath,{A.lib_path().parent}", "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    w, h, D = 120, 60, 40
    left, right = T.synthetic_pair(w, h, D, 91)
    left.tofile(tmp_path / "left.bgr"); right.tofile(tmp_path / "right.bgr")
    run = subprocess.run([str(exe), str(tmp_path / "left.bgr"), str(tmp_path / "right.bgr"), str(w), str(h), str(D),
                          str(tmp_path / "out")], capture_output=True, text=True, env=dict(os.environ, ADC_B200_QUIET="1"))
    assert run.returncode == 0 and "CONFIDENCE_OK" in run.stdout, (run.returncode, run.stdout[-500:], run.stderr[-500:])
    opt = T.default_option(max_disparity=D)
    want = GA.derive_aux(T.Oracle(w, h, opt), left, right, opt)
    for ext, key, dt in (("disp", "disp", np.float32), ("origin", "origin", np.uint8), ("best", "cost_best", np.float32),
                         ("second", "cost_second", np.float32)):
        _same(key, np.fromfile(tmp_path / f"out.{ext}", dt).reshape(h, w), want[key])
