"""Argument validation of the C ABI: which return code each entry point gives for a malformed design or batch.

Every case fails or returns before the first kernel launch.  The create functions check the whole design before
their first CUDA call, so those cases and the checks of the context-free entry points run without a GPU; the score
entry points of the PESQ, STOI, LSD and resampler contexts need a real context and are marked `gpu`."""
import ctypes

import numpy as np
import pytest

from fast_speech_enhancement_metrics_b200 import _lib, design

OK, INVALID = _lib.FSEM_OK, _lib.FSEM_E_INVALID
ROWS = 256                      # a non-null row address; no case gets far enough to read it
N_LIMIT = 1 << 30               # the device entry points take n < 2^30


def _last_error():
    return _lib.load().fsem_last_error().decode()


# ------------------------------------------------------------------ create functions
def _pesq_create(d):
    lib = _lib.load()
    handle = ctypes.c_void_p()
    rc = lib.fsem_pesq_create(ctypes.byref(handle), ctypes.byref(d))
    if handle.value:
        lib.fsem_pesq_destroy(handle)
    return rc


def test_pesq_create_rejects_a_wrong_taper():
    d, _ = design.pesq_design()
    d.taper[3] = 0.5
    assert _pesq_create(d) == INVALID
    assert "taper" in _last_error()


def test_pesq_create_rejects_a_broken_bark_band_layout():
    d, _ = design.pesq_design()
    d.band_first_bin[5] += 1
    assert _pesq_create(d) == INVALID
    assert "Bark band" in _last_error()


def test_pesq_create_rejects_a_negative_resampler_width():
    d, taps = design.pesq_design(8000)
    assert d.rs_orig != d.rs_neu and taps is not None
    d.rs_width = -1
    d.rs_ntaps = 2 * d.rs_width + d.rs_orig          # consistent tap count: the width alone is wrong
    assert _pesq_create(d) == INVALID
    assert "resampling kernel" in _last_error()


def test_stoi_create_rejects_bad_bands():
    lib = _lib.load()
    d, taps = design.stoi_design(16000)
    d.band_hi[3] = d.band_lo[3] - 1
    handle = ctypes.c_void_p()
    assert lib.fsem_stoi_create(ctypes.byref(handle), ctypes.byref(d)) == INVALID
    assert not handle.value and "band" in _last_error()


def test_resampler_create_rejects_a_negative_width():
    lib = _lib.load()
    taps = np.zeros(16, np.float32)
    handle = ctypes.c_void_p()
    rc = lib.fsem_resampler_create(ctypes.byref(handle), 2, 1, -1, 0, taps.ctypes.data_as(ctypes.POINTER(ctypes.c_float)))
    assert rc == INVALID
    assert not handle.value and "resampling kernel" in _last_error()


# ------------------------------------------------------------------ batch checks
# (batch, n, stride, rows) -> the code each entry point returns
SHAPES = {
    "empty_n0": (0, 0, 0, ROWS),
    "empty": (0, 16000, 16000, ROWS),
    "n_negative": (1, -1, 0, ROWS),
    "stride_below_n": (2, 16000, 8000, ROWS),
    "null_rows": (2, 16000, 16000, None),
    "n_2pow30": (1, N_LIMIT, N_LIMIT, ROWS),
}
# PESQ and STOI accept an empty batch whatever n is; LSD, SDR and the resampler reject n <= 0 even then
LENIENT_EMPTY = {"empty_n0": OK, "empty": OK, "n_negative": INVALID, "stride_below_n": INVALID,
                 "null_rows": INVALID, "n_2pow30": INVALID}
STRICT_N = dict(LENIENT_EMPTY, empty_n0=INVALID)


def _batch(name):
    b, n, stride, rows = SHAPES[name]
    return _lib.Batch(rows, rows, None, b, n, stride)


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_sdr_score_batch_checks(name):
    lib = _lib.load()
    batch = _batch(name)
    assert lib.fsem_sdr_score_f32(ctypes.byref(batch), ROWS, None, 0, None) == STRICT_N[name]


def test_sdr_score_rejects_more_than_65535_items():
    lib = _lib.load()
    batch = _lib.Batch(ROWS, ROWS, None, 65536, 16000, 16000)
    assert lib.fsem_sdr_score_f32(ctypes.byref(batch), ROWS, None, 0, None) == INVALID
    assert "65535" in _last_error()


# fsem_ingest_f32 has no upper bound on n, so an empty batch with n = 2^30 is accepted
INGEST = dict(LENIENT_EMPTY, n_2pow30=OK)


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_ingest_batch_checks(name):
    lib = _lib.load()
    b, n, stride, rows = SHAPES[name]
    if name == "n_2pow30":
        b = 0                                         # a non-empty batch of that size would be copied
    assert lib.fsem_ingest_f32(rows, _lib.DTYPE_F32, b, n, stride, ROWS, max(n, 0), None) == INGEST[name]


def test_ingest_rejects_a_destination_pitch_below_n():
    lib = _lib.load()
    assert lib.fsem_ingest_f32(ROWS, _lib.DTYPE_F32, 0, 16000, 16000, ROWS, 8000, None) == INVALID


def _null_context_calls(lib, batch):
    b = ctypes.byref(batch)
    return {
        "fsem_pesq_score": lambda: lib.fsem_pesq_score(None, b, _lib.DTYPE_F32, ROWS, None, None, 0, None),
        "fsem_stoi_score": lambda: lib.fsem_stoi_score(None, b, _lib.DTYPE_F32, ROWS, ROWS, None, None, None, 0, None),
        "fsem_lsd_score_f32": lambda: lib.fsem_lsd_score_f32(None, b, ROWS, None, 0, None),
        "fsem_resample_f32": lambda: lib.fsem_resample_f32(None, b, ROWS, 16000, None, None),
        "fsem_sdr_score_f32": lambda: lib.fsem_sdr_score_f32(None, ROWS, None, 0, None),
    }


@pytest.mark.parametrize("entry", ["fsem_pesq_score", "fsem_stoi_score", "fsem_lsd_score_f32", "fsem_resample_f32",
                                   "fsem_sdr_score_f32"])
def test_null_context_is_reported_under_the_called_name(entry):
    lib = _lib.load()
    batch = _lib.Batch(ROWS, ROWS, None, 4, 16000, 16000)
    assert _null_context_calls(lib, batch)[entry]() == INVALID
    assert _last_error().startswith(entry + ": null argument")


# ------------------------------------------------------------------ the same table with real contexts
@pytest.fixture(scope="module")
def contexts():
    from fast_speech_enhancement_metrics_b200 import LSD, PESQ, STOI
    return {"pesq": PESQ(16000), "stoi": STOI(16000), "lsd": LSD(16000), "lsd8k": LSD(8000)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SHAPES))
def test_device_entry_points_batch_checks(name, contexts):
    lib = _lib.load()
    batch = _batch(name)
    b = ctypes.byref(batch)
    pesq, stoi, lsd, rs = (contexts["pesq"]._ctx, contexts["stoi"]._ctx, contexts["lsd"]._ctx,
                           contexts["lsd8k"]._resampler)
    before = _lib.launch_count()
    assert lib.fsem_pesq_score(pesq, b, _lib.DTYPE_F32, ROWS, None, None, 0, None) == LENIENT_EMPTY[name]
    assert lib.fsem_stoi_score(stoi, b, _lib.DTYPE_F32, ROWS, ROWS, None, None, None, 0, None) == LENIENT_EMPTY[name]
    assert lib.fsem_lsd_score_f32(lsd, b, ROWS, None, 0, None) == STRICT_N[name]
    assert lib.fsem_resample_f32(rs, b, ROWS, max(SHAPES[name][1], 0), None, None) == STRICT_N[name]
    assert _lib.launch_count() == before
