"""STOI / ESTOI with 10 kHz resample-on-ingest and silent-frame removal, drop-in for
fast_se_metrics.STOI.

Same constructor and call contract as fast_se_metrics/STOI.py:7-205:
`STOI(sample_rate=10000, use_gpu=False)(clean, denoised) -> [{"STOI": f, "ESTOI": f}, ...]`.
"""
from __future__ import annotations

import ctypes as C
import warnings

import torch

from . import _lib
from .base import BaseMetric, make_batch, score_host, stream_ptr
from .design import stoi_design


class STOI(BaseMetric):
    higher_is_better = True
    EXPECTED_SAMPLING_RATE = 10000

    def __init__(self, sample_rate: int = 10000, use_gpu: bool = False):
        super().__init__(sample_rate, use_gpu)
        self.N = 30
        self._design, self._taps = stoi_design(self.sample_rate, self.EXPECTED_SAMPLING_RATE)
        handle = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.fsem_stoi_create(C.byref(handle), C.byref(self._design)))
        self._ctx = handle

    def __del__(self):
        ctx = getattr(self, "_ctx", None)
        if ctx is not None and ctx.value:
            try:
                self._lib.fsem_stoi_destroy(ctx)
            except Exception:
                pass
            self._ctx = None

    # ------------------------------------------------------------------
    def score_tensors(self, clean: torch.Tensor, deg: torch.Tensor, lengths=None):
        """Device-resident scoring: returns (scores[2, B] f32 = STOI row 0 / ESTOI row 1, kept[B] i32,
        status[B] i32) CUDA tensors, stream-ordered, no host synchronisation."""
        clean, deg = self._on_device(clean), self._on_device(deg)
        b, n = clean.shape
        lens = self._lengths_tensor(lengths, b, n, clean.device)
        scores = torch.empty(2, b, dtype=torch.float32, device=clean.device)
        kept = torch.empty(b, dtype=torch.int32, device=clean.device)
        status = torch.empty(b, dtype=torch.int32, device=clean.device)
        batch, clean, deg = make_batch(clean, deg, lens)
        with torch.cuda.device(clean.device):
            ws = self._get_workspace(self._lib.fsem_stoi_workspace_bytes(self._ctx, b, n))
            _lib.check(self._lib.fsem_stoi_score(
                self._ctx, C.byref(batch), _lib.dtype_code(clean.dtype), scores[0].data_ptr(), scores[1].data_ptr(), kept.data_ptr(),
                status.data_ptr(), ws.data_ptr(), ws.numel(), stream_ptr(clean.device)))
        self._last_shape = (b, n)
        self._last_lengths = lens
        return scores, kept, status

    def mask_margin(self) -> torch.Tensor:
        """After a device-resident score call: margin[B] (CUDA, dB) = min over the item's analysis frames of
        |(max E - 40) - E_t|, i.e. how far the closest frame was from flipping the keep/drop decision of
        STOI.py:98-102.  The mask is bit-exact against any fp32 evaluation of the frame norm whenever the
        margin exceeds the norm's rounding noise (~1e-6 dB); ties are reported by this margin, not hidden."""
        b, n = self._last_shape
        lens = getattr(self, "_last_lengths", None)
        out = torch.empty(b, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.fsem_stoi_mask_margin(
                self._ctx, b, n, lens.data_ptr() if lens is not None else None, self._workspace.data_ptr(),
                out.data_ptr(), stream_ptr(self.device)))
        return out

    def score_host(self, clean: torch.Tensor, deg: torch.Tensor, lengths=None):
        """Host-resident scoring: CPU [B, n] float32 / int16 / float16 tensors in, CPU tensors out."""
        _, _, scores, kept, status = score_host(None, self, clean, deg, lengths)
        return scores, kept, status

    def compute_metric(self, clean_speech, denoised_speech, lengths=None) -> list[dict[str, float]]:
        assert clean_speech is not None                                   # STOI.py:203
        if clean_speech.is_cuda:
            scores, kept, _ = self.score_tensors(clean_speech, denoised_speech, lengths)
            packed = torch.cat([scores, kept.to(torch.float32)[None]]).cpu()   # ONE device->host copy
            scores, kept = packed[:2], packed[2].to(torch.int32)
        else:
            scores, kept, _ = self.score_host(clean_speech, denoised_speech, lengths)
        self.last_kept_frames = kept
        if int(kept.max()) <= self.N + 1:
            # no 30-frame segment in the whole batch: the reference warns, returns 0-d tensors and
            # then fails in zip() with TypeError (STOI.py:163-165, 205)
            warnings.warn("Not enough non-silent frames. Please check your sound files", RuntimeWarning, stacklevel=2)
            raise TypeError("iteration over a 0-d tensor")
        return [{"STOI": s, "ESTOI": e} for s, e in zip(scores[0].tolist(), scores[1].tolist())]

    # ------------------------------------------------------------------ stage taps (tests)
    def debug_taps(self):
        """After score_tensors: dict(mask[B, words] int32 bit t = frame t kept,
        tob[2, B, 15, U], resampled[2, B, L] or None)."""
        b, n = self._last_shape
        dims = (C.c_int64 * 3)()
        with torch.cuda.device(self.device):
            stream = stream_ptr(self.device)
            ws = self._workspace.data_ptr()
            _lib.check(self._lib.fsem_stoi_debug_taps(self._ctx, b, n, ws, None, None, None, dims, stream))
            mask = torch.empty(b, dims[0], dtype=torch.int32, device=self.device)
            tob = torch.empty(2, b, 15, dims[1], dtype=torch.float32, device=self.device)
            res = torch.empty(2, b, dims[2], dtype=torch.float32, device=self.device) if dims[2] else None
            _lib.check(self._lib.fsem_stoi_debug_taps(self._ctx, b, n, ws, mask.data_ptr(), tob.data_ptr(),
                                                      res.data_ptr() if res is not None else None, dims, stream))
        return {"mask": mask, "tob": tob, "resampled": res}
