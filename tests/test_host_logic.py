"""CPU tests (-m "not gpu"): host-side design code, the C-ABI library's exports, and the
shape arithmetic shared by host and device.  No compute calls (there is no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest
from scipy.signal import lfilter

from fast_speech_enhancement_metrics_b200 import _lib, design, p862_tables
from oracle import pesq_oracle as po
from oracle import stoi_oracle as so
from oracle import tables as otab
from tests.conftest import ROOT


def test_library_loads_and_exports_every_declared_symbol():
    lib = _lib.load()
    assert lib.fsem_version() == 200
    header = open(os.path.join(ROOT, "include", "fsem.h")).read()
    declared = set(re.findall(r"FSEM_API [^;(]*?\b(fsem_[a-z0-9_]+)\(", header))
    assert declared == set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(lib, name)
    assert lib.fsem_last_error() is not None


def test_struct_layouts_match_header_sizes():
    # sizes implied by include/fsem.h (all members are 4-byte scalars except the taps pointer)
    assert ctypes.sizeof(design.PesqDesign) == 4 * (1 + 4 * 5 + 3 + 2 + 15 + 1 + 512 + 6 * 49 + 1) + 4 * 4 + 4 + 8   # + resampler, pad, taps*
    assert ctypes.sizeof(design.StoiDesign) == 16 + 8 + 4 * 256 + 4 * 30 + 8
    assert ctypes.sizeof(_lib.Batch) == 48


def test_tables_agree_with_oracle_copy():
    assert np.array_equal(p862_tables.BINS_PER_BAND, otab.BINS_PER_BAND)
    assert np.array_equal(p862_tables.CENTRE_BARK, otab.BAND_CENTRE_BARK)
    assert np.array_equal(p862_tables.WIDTH_BARK, otab.BAND_WIDTH_BARK)
    assert np.array_equal(p862_tables.POW_DENS_CORRECTION, otab.POWER_DENSITY_CORRECTION)
    assert np.array_equal(p862_tables.ABS_THRESH_POWER, otab.ABS_THRESHOLD_POWER)


def test_pesq_design_reproduces_the_reference_filter(golden_pesq):
    b32, a32 = design.power_filter_f32()
    assert np.array_equal(b32, golden_pesq["tap_power_filter"][0])
    assert np.array_equal(a32, golden_pesq["tap_power_filter"][1])
    d, _ = design.pesq_design()
    assert np.array_equal(np.array(d.hann[:], np.float32), golden_pesq["tap_hann512"])
    # the float32 parallel form run in float64 reproduces the direct form's band power
    rng = np.random.default_rng(0)
    x = lfilter([1.0], [1.0, -0.97], rng.standard_normal(20000))
    y = d.bp_direct * x
    for s in range(5):
        y = y + lfilter([d.bp_c0[s], d.bp_c1[s]], [1.0, d.bp_a1[s], d.bp_a2[s]], x)
    p_ref = po.band_power(x)
    assert abs(np.dot(y, y) - p_ref) <= 2e-5 * p_ref
    assert d.warmup % 64 == 0 and 512 <= d.warmup <= 1024
    assert list(d.band_first_bin[:3]) == [0, 1, 2] and d.band_first_bin[48] + d.band_num_bins[48] == 256


def test_stoi_design_matches_reference_constants(golden_stoi):
    d, taps = design.stoi_design(16000)
    assert (d.orig, d.neu, d.width, d.ntaps) == (8, 5, 10, 28)
    assert np.array_equal(taps, golden_stoi["tap_resample_kernel"])
    assert np.array_equal(np.array(d.window[:], np.float32), golden_stoi["tap_window"])
    obm = np.zeros((15, 257), np.float32)
    for i in range(15):
        obm[i, d.band_lo[i]:d.band_hi[i]] = 1
    assert np.array_equal(obm, golden_stoi["tap_obm"])
    d10, taps10 = design.stoi_design(10000)
    assert d10.orig == d10.neu and taps10 is None
    t, w, o, n = design.sinc_hann_kernel(8000, 10000)
    ot, ow, oo, on = so.resample_kernel(8000, 10000)
    assert (w, o, n) == (ow, oo, on) and np.array_equal(t, ot)


def test_metric_constructor_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from fast_speech_enhancement_metrics_b200 import PESQ, STOI
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        PESQ(16000, use_gpu=True)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        STOI(16000, use_gpu=False)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "fast_speech_enhancement_metrics_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, re.M), f
                assert "/root/reference" not in text, f


def test_ingest_dtype_codes_follow_the_header():
    """FSEM_DTYPE_* in include/fsem.h <-> _lib.dtype_code; unsupported dtypes fail like the reference
    (float64 raises "expected scalar type Float" inside lfilter / stft there)."""
    import re
    import torch
    from fast_speech_enhancement_metrics_b200 import _lib
    header = open(os.path.join(ROOT, "include", "fsem.h")).read()
    codes = {name: int(val) for name, val in re.findall(r"#define FSEM_DTYPE_(\w+) (\d+)", header)}
    assert codes == {"F32": _lib.DTYPE_F32, "I16": _lib.DTYPE_I16, "F16": _lib.DTYPE_F16}
    assert _lib.dtype_code(torch.float32) == codes["F32"]
    assert _lib.dtype_code(torch.int16) == codes["I16"]
    assert _lib.dtype_code(torch.float16) == codes["F16"]
    for bad in (torch.float64, torch.int32, torch.bfloat16):
        with pytest.raises(RuntimeError, match="expected scalar type Float"):
            _lib.dtype_code(bad)


def test_graph_entry_points_validate_their_arguments_without_a_gpu():
    """fsem_graph_*: argument validation comes before any CUDA call, so it can be checked here (no compute)."""
    lib = _lib.load()
    handle = ctypes.c_void_p()
    batch = _lib.Batch(None, None, None, 4, 16000, 16000)
    assert lib.fsem_graph_create(ctypes.byref(handle), None, None, ctypes.byref(batch), _lib.DTYPE_F32,
                                 None, None, None, None, None, None, 1) == _lib.FSEM_E_INVALID
    assert b"no metric" in lib.fsem_last_error()
    assert not handle.value
    assert lib.fsem_graph_create(None, None, None, ctypes.byref(batch), _lib.DTYPE_F32,
                                 None, None, None, None, None, None, 1) == _lib.FSEM_E_INVALID
    assert lib.fsem_graph_launch(None, None) == _lib.FSEM_E_INVALID
    assert lib.fsem_graph_nodes(None) == 0 and lib.fsem_graph_slices(None) == 0
    assert lib.fsem_graph_destroy(None) == _lib.FSEM_OK


_C_CONSUMER = r"""
#include <stddef.h>
#include <stdio.h>
#include <string.h>
#include "fsem.h"
int main(void) {
    fsem_batch_t b;
    memset(&b, 0, sizeof b);
    printf("batch %zu %zu %zu %zu %zu %zu %zu\n", sizeof(fsem_batch_t), offsetof(fsem_batch_t, clean), offsetof(fsem_batch_t, deg),
           offsetof(fsem_batch_t, lengths), offsetof(fsem_batch_t, batch), offsetof(fsem_batch_t, n), offsetof(fsem_batch_t, stride));
    printf("pesq %zu %zu %zu %zu %zu\n", sizeof(fsem_pesq_design_t), offsetof(fsem_pesq_design_t, hann),
           offsetof(fsem_pesq_design_t, band_first_bin), offsetof(fsem_pesq_design_t, sl), offsetof(fsem_pesq_design_t, rs_taps));
    printf("stoi %zu %zu %zu %zu %zu\n", sizeof(fsem_stoi_design_t), offsetof(fsem_stoi_design_t, taps),
           offsetof(fsem_stoi_design_t, window), offsetof(fsem_stoi_design_t, band_lo), offsetof(fsem_stoi_design_t, dyn_range));
    printf("version %d %d\n", fsem_version(), FSEM_VERSION);
    /* argument validation happens before any CUDA call: a C caller gets the error code and the message */
    printf("null %d %s\n", fsem_pesq_score(NULL, &b, FSEM_DTYPE_F32, NULL, NULL, NULL, 0, NULL), fsem_last_error());
    printf("ws %zu\n", fsem_sdr_workspace_bytes(0, 0));
    return 0;
}
"""


def test_header_is_plain_c_and_a_c_program_can_call_the_library(tmp_path):
    """The drop-in boundary is a C ABI: include/fsem.h must compile as C99 (gcc -std=c99 -pedantic-errors), a C program
    must link against the built library, and the struct layouts the C compiler sees must be the ones the Python mirror
    (ctypes) uses.  No compute call (no GPU here): version, argument validation, a workspace query."""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    lib_dir = os.path.dirname(_lib.LIB_PATH)
    src = tmp_path / "consumer.c"
    src.write_text(_C_CONSUMER)
    exe = tmp_path / "consumer"
    subprocess.run([gcc, "-std=c99", "-pedantic-errors", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                    "-o", str(exe), "-L", lib_dir, "-l:" + os.path.basename(_lib.LIB_PATH), "-Wl,-rpath," + lib_dir],
                   check=True, capture_output=True, text=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines()
    rows = {ln.split()[0]: ln.split()[1:] for ln in out}
    B, P, S = _lib.Batch, design.PesqDesign, design.StoiDesign
    assert [int(v) for v in rows["batch"]] == [ctypes.sizeof(B), B.clean.offset, B.deg.offset, B.lengths.offset,
                                               B.batch.offset, B.n.offset, B.stride.offset]
    assert [int(v) for v in rows["pesq"]] == [ctypes.sizeof(P), P.hann.offset, P.band_first_bin.offset, P.sl.offset,
                                              P.rs_taps.offset]
    assert [int(v) for v in rows["stoi"]] == [ctypes.sizeof(S), S.taps.offset, S.window.offset, S.band_lo.offset,
                                              S.dyn_range.offset]
    assert rows["version"] == ["200", "200"]
    assert int(rows["null"][0]) == -1 and len(rows["null"]) > 1          # FSEM_E_INVALID + a message
    assert rows["ws"] == ["0"]


def test_bench_dump_outputs_writes_float32_columns_and_samples_above_the_limit(tmp_path, monkeypatch):
    import bench
    table = np.arange(30, dtype=np.float32).reshape(10, 3)
    bench.dump_outputs(str(tmp_path / "all"), table)
    assert sorted(os.listdir(tmp_path / "all")) == ["estoi.npy", "pesq.npy", "stoi.npy"]
    for j, name in enumerate(("pesq", "stoi", "estoi")):
        col = np.load(tmp_path / "all" / (name + ".npy"))
        assert col.dtype == np.float32 and np.array_equal(col, table[:, j])
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4 * (3 * 4 + 8))      # room for 4 rows and their indices
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), table)
    idx = np.load(tmp_path / "a" / "items.npy")
    assert idx.dtype == np.float64 and len(idx) == 4 and np.array_equal(idx, np.load(tmp_path / "b" / "items.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "stoi.npy"), table[idx.astype(int), 1])
    assert sum(f.stat().st_size - 128 for f in (tmp_path / "a").iterdir()) <= bench.DUMP_LIMIT_BYTES   # 128: .npy header


def test_bench_rejects_zero_timed_steps():
    import subprocess
    import sys
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert res.returncode == 2 and "--steps must be at least 1" in res.stderr
