"""Wide-band PESQ (no time alignment), drop-in for fast_se_metrics.PESQ.

Same constructor and call contract as fast_se_metrics/PESQ.py:13-245:
`PESQ(sample_rate=16000, use_gpu=False)(clean, denoised) -> [{"PESQ": float}, ...]`.
All arithmetic of PESQ.compute_metric runs in libfsem_b200.so (three CUDA kernels).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from .base import BaseMetric, check_score, make_batch, score_host, stream_ptr
from .design import pesq_design


class PESQ(BaseMetric):
    higher_is_better = True
    EXPECTED_SAMPLING_RATE = 16000

    def __init__(self, sample_rate: int = 16000, use_gpu: bool = False):
        super().__init__(sample_rate, use_gpu)
        # resample-on-ingest (base.py:13,19-20) runs inside the library as its first kernel
        self._design, self._taps = pesq_design(self.sample_rate, self.EXPECTED_SAMPLING_RATE)
        handle = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.fsem_pesq_create(C.byref(handle), C.byref(self._design)))
        self._ctx = handle

    def __del__(self):
        ctx = getattr(self, "_ctx", None)
        if ctx is not None and ctx.value:
            try:
                self._lib.fsem_pesq_destroy(ctx)
            except Exception:
                pass
            self._ctx = None

    # ------------------------------------------------------------------
    def score_tensors(self, clean: torch.Tensor, deg: torch.Tensor, lengths=None):
        """Device-resident scoring: returns (mos[B] f32, status[B] i32) CUDA tensors, stream-ordered,
        no host synchronisation.  `clean`/`deg` are [B, n] float32 / int16 / float16 CUDA tensors (the IIR pass reads
        them in their own dtype: fsem_pesq_score)."""
        clean, deg = self._on_device(clean), self._on_device(deg)
        b, n = clean.shape
        lens = self._lengths_tensor(lengths, b, n, clean.device)
        mos = torch.empty(b, dtype=torch.float32, device=clean.device)
        status = torch.empty(b, dtype=torch.int32, device=clean.device)
        batch, clean, deg = make_batch(clean, deg, lens)
        with torch.cuda.device(clean.device):
            ws = self._get_workspace(self._lib.fsem_pesq_workspace_bytes(self._ctx, b, n))
            check_score(self._lib.fsem_pesq_score(
                self._ctx, C.byref(batch), _lib.dtype_code(clean.dtype), mos.data_ptr(), status.data_ptr(), ws.data_ptr(),
                ws.numel(), stream_ptr(clean.device)))
        self._last_shape = (b, n)
        return mos, status

    def score_host(self, clean: torch.Tensor, deg: torch.Tensor, lengths=None):
        """Host-resident scoring: CPU [B, n] float32 / int16 / float16 tensors in, CPU tensors out; the
        library overlaps the host->device copies with compute."""
        mos, status, _, _, _ = score_host(self, None, clean, deg, lengths)
        return mos, status

    def compute_metric(self, clean_speech, denoised_speech, lengths=None) -> list[dict[str, float]]:
        assert clean_speech is not None                                   # PESQ.py:235
        if clean_speech.is_cuda:
            mos, status = self.score_tensors(clean_speech, denoised_speech, lengths)
            both = torch.stack([mos, status.to(torch.float32)]).cpu()    # ONE device->host copy
            mos, status = both[0], both[1].to(torch.int32)
        else:
            mos, status = self.score_host(clean_speech, denoised_speech, lengths)
        if lengths is not None and bool((status == _lib.ITEM_TOO_SHORT).any()):
            raise RuntimeError("PESQ needs at least 20 frames of 512/256 samples for every item")
        return [{"PESQ": m} for m in mos.tolist()]                       # PESQ.py:245

    # ------------------------------------------------------------------ stage taps (tests)
    def debug_taps(self):
        """After score_tensors: (bark[2, B, T, 49] level-aligned Bark power densities,
        band_power[2, B] float64 sums of y^2 of the band-passed inputs)."""
        b, n = self._last_shape
        frames = C.c_int64()
        with torch.cuda.device(self.device):
            stream = stream_ptr(self.device)
            _lib.check(self._lib.fsem_pesq_debug_taps(self._ctx, b, n, self._workspace.data_ptr(), None, None,
                                                      C.byref(frames), stream))
            bark = torch.empty(2, b, frames.value, 49, dtype=torch.float32, device=self.device)
            power = torch.empty(2, b, dtype=torch.float64, device=self.device)
            _lib.check(self._lib.fsem_pesq_debug_taps(self._ctx, b, n, self._workspace.data_ptr(), bark.data_ptr(),
                                                      power.data_ptr(), C.byref(frames), stream))
        return bark, power
