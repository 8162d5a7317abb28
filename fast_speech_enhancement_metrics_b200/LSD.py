"""Log-spectral distance, drop-in for fast_se_metrics.LSD (SURVEY.md 8f rank 3: an adjacent metric that
reuses the packed warp FFT).  Same contract as fast_se_metrics/LSD.py:6-52:
`LSD(sample_rate=16000, use_gpu=False)(clean, denoised) -> [{"LSD": float}, ...]`, lower is better."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from .base import BaseMetric, make_batch, stream_ptr


class LSD(BaseMetric):
    higher_is_better = False
    EXPECTED_SAMPLING_RATE = 16000

    def __init__(self, sample_rate: int = 16000, use_gpu: bool = False):
        super().__init__(sample_rate, use_gpu)
        self._make_resampler()                                              # base.py:13 (None at 16 kHz)
        self.nfft, self.hop = 512, 256                                      # LSD.py:12-13
        window = torch.hann_window(self.nfft, dtype=torch.float32)          # LSD.py:16
        self._window = (C.c_float * 512)(*window.tolist())
        handle = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.fsem_lsd_create(C.byref(handle), self._window))
        self._ctx = handle

    def __del__(self):
        ctx = getattr(self, "_ctx", None)
        if ctx is not None and ctx.value:
            try:
                self._lib.fsem_lsd_destroy(ctx)
            except Exception:
                pass
            self._ctx = None
        self._free_resampler()

    def score_tensors(self, clean: torch.Tensor, deg: torch.Tensor, lengths=None) -> torch.Tensor:
        """[B, n] float32 CUDA tensors -> lsd[B] CUDA tensor, stream-ordered, no host synchronisation."""
        clean, deg = self._as_f32(self._on_device(clean)), self._as_f32(self._on_device(deg))
        b, n = clean.shape
        lens = self._lengths_tensor(lengths, b, n, clean.device)
        clean, deg, lens = self._resample_pair(clean, deg, lens)            # base.py:19-20
        b, n = clean.shape
        out = torch.empty(b, dtype=torch.float32, device=clean.device)
        batch, clean, deg = make_batch(clean, deg, lens)
        with torch.cuda.device(clean.device):
            ws = self._get_workspace(self._lib.fsem_lsd_workspace_bytes(self._ctx, b, n))
            _lib.check(self._lib.fsem_lsd_score_f32(self._ctx, C.byref(batch), out.data_ptr(), ws.data_ptr(), ws.numel(),
                                                    stream_ptr(clean.device)))
        return out

    def compute_metric(self, clean_speech, denoised_speech, lengths=None) -> list[dict[str, float]]:
        assert clean_speech is not None                                     # LSD.py:36
        if not clean_speech.is_cuda:                                        # host tensors (base.py:18): chunked uploads
            return [{"LSD": v} for v in self._score_host_overlapped(clean_speech, denoised_speech, lengths).tolist()]
        return [{"LSD": v} for v in self.score_tensors(clean_speech, denoised_speech, lengths).cpu().tolist()]
