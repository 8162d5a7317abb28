"""Signal-to-distortion ratio (512-tap distortion filter), drop-in for fast_se_metrics.SDR (SURVEY.md 8f rank 3).
Same contract as fast_se_metrics/SDR.py:52-97: `SDR(sample_rate=16000, use_gpu=False)(clean, denoised) ->
[{"SDR": float}, ...]` in dB, higher is better."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from .base import BaseMetric, make_batch, stream_ptr


class SDR(BaseMetric):
    higher_is_better = True
    EXPECTED_SAMPLING_RATE = 16000

    def __init__(self, sample_rate: int = 16000, use_gpu: bool = False):
        super().__init__(sample_rate, use_gpu)
        self._make_resampler()                                               # base.py:13 (None at 16 kHz)
        self.filter_length = 512                                             # SDR.py:58

    def __del__(self):
        self._free_resampler()

    def score_tensors(self, clean: torch.Tensor, deg: torch.Tensor, lengths=None) -> torch.Tensor:
        """[B, n] float32 CUDA tensors -> sdr[B] (dB) CUDA tensor, stream-ordered, no host synchronisation."""
        clean, deg = self._as_f32(self._on_device(clean)), self._as_f32(self._on_device(deg))
        b, n = clean.shape
        lens = self._lengths_tensor(lengths, b, n, clean.device)
        clean, deg, lens = self._resample_pair(clean, deg, lens)             # base.py:19-20
        b, n = clean.shape
        out = torch.empty(b, dtype=torch.float32, device=clean.device)
        batch, clean, deg = make_batch(clean, deg, lens)
        with torch.cuda.device(clean.device):
            ws = self._get_workspace(self._lib.fsem_sdr_workspace_bytes(b, n))
            _lib.check(self._lib.fsem_sdr_score_f32(C.byref(batch), out.data_ptr(), ws.data_ptr(), ws.numel(),
                                                    stream_ptr(clean.device)))
        return out

    def compute_metric(self, clean_speech, denoised_speech, lengths=None) -> list[dict[str, float]]:
        assert clean_speech is not None                                      # SDR.py:75
        if not clean_speech.is_cuda:                                        # host tensors (base.py:18): chunked uploads
            return [{"SDR": v} for v in self._score_host_overlapped(clean_speech, denoised_speech, lengths).tolist()]
        return [{"SDR": v} for v in self.score_tensors(clean_speech, denoised_speech, lengths).cpu().tolist()]
