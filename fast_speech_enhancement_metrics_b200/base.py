"""Common base of the metric classes: argument checking, batching and dispatch.

Mirrors fast_se_metrics/base.py:6-43 (`BaseMetric(sample_rate, use_gpu)`,
`prepare_audio`, `prepare_inputs`, `compute_metric`, `__call__`).  Differences,
all deliberate:

* the arithmetic always runs on the current CUDA device through libfsem_b200.so;
  `use_gpu` is kept for signature compatibility and only records where the caller
  expects to hand tensors over (CPU tensors go through the library's host entry
  point, which overlaps the host->device copy with compute; CUDA tensors are
  consumed in place on the current stream).  Without a CUDA device or without the
  built library the constructor raises -- there is no CPU fallback;
* resample-on-ingest (base.py:19-20) is not a separate torchaudio op: STOI fuses
  it into its first kernel;
* optional `lengths=` (per-item valid samples of a padded batch); `None` gives
  exactly the reference behaviour;
* ingest formats (SURVEY.md 8f rank 2): besides float32, int16 PCM and float16 tensors are accepted and
  widened to float32 on the device with a value-preserving cast (bit-identical scores to `x.float()`); a CPU
  batch then crosses PCIe at 2 bytes per sample.  Anything else raises like the reference.
"""
from __future__ import annotations

import ctypes as C
from abc import ABC, abstractmethod

import torch

from . import _lib


def stream_ptr(device) -> C.c_void_p:
    """The current CUDA stream of `device` as the library's `void* stream` argument."""
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _ptr(t):
    return t.data_ptr() if t is not None else None


def make_batch(clean: torch.Tensor, deg: torch.Tensor, lens):
    """[B, n] clean / deg rows and optional int32 lengths[B] -> (_lib.Batch, clean, deg).  The library takes one row
    pitch for both signals, so rows of different pitch are made contiguous; the returned tensors are the ones the
    struct points at and must stay alive for the call."""
    b, n = clean.shape
    if deg.stride(0) != clean.stride(0) and b > 1:
        clean, deg = clean.contiguous(), deg.contiguous()
    batch = _lib.Batch(clean.data_ptr(), deg.data_ptr(), _ptr(lens), b, n,
                       clean.stride(0) if b > 1 else max(n, clean.stride(0)))
    return batch, clean, deg


def check_score(code: int) -> None:
    if code == _lib.FSEM_E_TOO_SHORT:
        # the reference's unfold(1, size=20, step=10) fails the same way (PESQ.py:169)
        raise RuntimeError(_lib.load().fsem_last_error().decode())
    _lib.check(code)


def score_host(pesq, stoi, clean: torch.Tensor, deg: torch.Tensor, lengths=None):
    """Host-resident scoring of PESQ, STOI or both on one upload (fsem_score_host): CPU [B, n] float32 / int16 /
    float16 rows in, CPU tensors out: (mos[B], pesq_status[B], scores[2, B] = STOI / ESTOI rows, kept[B],
    stoi_status[B]), None for the outputs of a metric that is None.  The library overlaps the host->device copies
    with compute."""
    owner = pesq if pesq is not None else stoi
    b, n = clean.shape
    lens = BaseMetric._lengths_tensor(lengths, b, n, "cpu")
    batch, clean, deg = make_batch(clean, deg, lens)
    mos = pst = scores = kept = sst = None
    if pesq is not None:
        mos, pst = torch.empty(b, dtype=torch.float32), torch.empty(b, dtype=torch.int32)
    if stoi is not None:
        scores = torch.empty(2, b, dtype=torch.float32)
        kept, sst = torch.empty(b, dtype=torch.int32), torch.empty(b, dtype=torch.int32)
    with torch.cuda.device(owner.device):
        check_score(owner._lib.fsem_score_host(
            pesq._ctx if pesq is not None else None, stoi._ctx if stoi is not None else None, batch.clean, batch.deg,
            _lib.dtype_code(clean.dtype), batch.lengths, b, n, batch.stride, _ptr(mos), _ptr(pst),
            _ptr(None if scores is None else scores[0]), _ptr(None if scores is None else scores[1]), _ptr(kept),
            _ptr(sst)))
    return mos, pst, scores, kept, sst


class BaseMetric(ABC):
    higher_is_better: bool
    EXPECTED_SAMPLING_RATE: int

    def __init__(self, sample_rate: int = 16000, use_gpu: bool = False):
        self.sample_rate = int(sample_rate)
        self.use_gpu = bool(use_gpu)
        self._lib = _lib.load()                       # raises ImportError if the .so is missing
        if not torch.cuda.is_available():
            raise RuntimeError("fast_speech_enhancement_metrics_b200 needs a CUDA device (sm_100a); "
                               "there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device())
        self._workspace = None

    # ------------------------------------------------------------------ reference API
    def prepare_audio(self, audio: torch.Tensor) -> torch.Tensor:
        """base.py:16-21: at least 2-D, unit stride along time.  The tensor stays where it is (no
        implicit device move for CPU tensors); inputs are never modified and keep their dtype: float32, int16 PCM and
        float16 rows are all consumed in place by the first kernel of the metric."""
        audio = torch.atleast_2d(audio)
        if audio.dim() != 2:
            raise Exception("expected a [batch, samples] tensor")
        _lib.dtype_code(audio.dtype)                  # raises for float64 & co like the reference
        if audio.stride(1) != 1 or (audio.shape[0] > 1 and audio.stride(0) < audio.shape[1]):
            audio = audio.contiguous()
        return self._on_device(audio)

    def _as_f32(self, audio: torch.Tensor) -> torch.Tensor:
        """float32 CUDA rows for the kernels that only read float32 (LSD, SDR, the general resampler building block):
        int16 / float16 CUDA tensors are widened with fsem_ingest_f32.  PESQ and STOI do not need this: their first
        kernels read int16 / float16 rows directly (fsem_pesq_score / fsem_stoi_score)."""
        code = _lib.dtype_code(audio.dtype)
        return audio if code == _lib.DTYPE_F32 else self._ingest(audio, code)

    def _on_device(self, audio: torch.Tensor) -> torch.Tensor:
        """The context tables, resampler taps and workspace of a metric live on the device that was current at
        construction (self.device).  A CUDA tensor on ANOTHER device is moved there, as the reference's
        prepare_audio does with `.to(self.device)` (base.py:18); CPU tensors stay on the host for the library's
        overlapped upload."""
        if audio.is_cuda and audio.device != self.device:
            audio = audio.to(self.device)
        return audio

    def _ingest(self, audio: torch.Tensor, code: int) -> torch.Tensor:
        b, n = audio.shape
        out = torch.empty(b, (n + 3) // 4 * 4, dtype=torch.float32, device=audio.device)[:, :n]
        if b and n:
            with torch.cuda.device(audio.device):
                _lib.check(self._lib.fsem_ingest_f32(
                    audio.data_ptr(), code, b, n, audio.stride(0) if b > 1 else max(n, audio.stride(0)),
                    out.data_ptr(), out.stride(0), stream_ptr(audio.device)))
        return out

    def prepare_inputs(self, clean_speech, denoised_speech):
        if clean_speech is not None and clean_speech.shape != denoised_speech.shape:
            raise Exception("`clean_speech` and `denoised_speech` should have the same shape.")   # base.py:26-27
        if clean_speech is not None:
            clean_speech = self.prepare_audio(clean_speech)
        denoised_speech = self.prepare_audio(denoised_speech)
        if clean_speech is not None and clean_speech.device != denoised_speech.device:
            raise Exception("`clean_speech` and `denoised_speech` should be on the same device.")
        if clean_speech is not None and clean_speech.dtype != denoised_speech.dtype:
            raise Exception("`clean_speech` and `denoised_speech` should have the same dtype.")
        return clean_speech, denoised_speech

    @abstractmethod
    def compute_metric(self, clean_speech, denoised_speech, lengths=None) -> list[dict[str, float]]:
        raise NotImplementedError

    def __call__(self, clean_speech, denoised_speech, lengths=None) -> list[dict[str, float]]:
        clean_speech, denoised_speech = self.prepare_inputs(clean_speech, denoised_speech)
        return self.compute_metric(clean_speech, denoised_speech, lengths)

    # ------------------------------------------------------------------ resample-on-ingest (base.py:13,19-20)
    def _make_resampler(self):
        """For metrics that do not fuse the resampling into their own first kernel (LSD, SDR): a library
        resampler context holding torchaudio's sinc-Hann kernel for sample_rate -> EXPECTED_SAMPLING_RATE."""
        from .design import sinc_hann_kernel
        self._resampler = None
        if self.sample_rate == self.EXPECTED_SAMPLING_RATE:
            return
        taps, width, o, nw = sinc_hann_kernel(self.sample_rate, self.EXPECTED_SAMPLING_RATE)
        handle = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.fsem_resampler_create(C.byref(handle), o, nw, width, taps.shape[1],
                                                       taps.ctypes.data_as(C.POINTER(C.c_float))))
        self._resampler = handle

    def _free_resampler(self):
        r = getattr(self, "_resampler", None)
        if r is not None and r.value:
            try:
                self._lib.fsem_resampler_destroy(r)
            except Exception:
                pass
        self._resampler = None

    def _resample_pair(self, clean: torch.Tensor, deg: torch.Tensor, lens):
        """[B, n] float32 CUDA rows at sample_rate -> ([B, L] clean, [B, L] deg, lengths or None) at the expected
        rate, one kernel launch for both signals (fsem_resample_f32)."""
        if getattr(self, "_resampler", None) is None:
            return clean, deg, lens
        b, n = clean.shape
        L = int(self._lib.fsem_resampled_len(self._resampler, n))
        pitch = (L + 3) // 4 * 4
        out = torch.empty(2, b, pitch, dtype=torch.float32, device=self.device)
        new_lens = torch.empty(b, dtype=torch.int32, device=self.device) if lens is not None else None
        batch, clean, deg = make_batch(clean, deg, lens)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.fsem_resample_f32(self._resampler, C.byref(batch), out.data_ptr(), pitch, _ptr(new_lens),
                                                   stream_ptr(self.device)))
        return out[0, :, :L], out[1, :, :L], new_lens

    def _score_host_overlapped(self, clean: torch.Tensor, deg: torch.Tensor, lengths=None) -> torch.Tensor:
        """Host rows -> per-item scores (CPU tensor) for the metrics whose library entry point is device-only (LSD,
        SDR): the batch is cut into chunks of ~128 MB, chunk k + 1 is uploaded on a copy stream while chunk k is
        scored on the current stream (the same double-buffered scheme as the library's fsem_score_host pipeline for
        PESQ / STOI), and all scores come back in ONE device->host copy.  Needs pinned host tensors to overlap;
        pageable ones still work, serialised by the driver."""
        b, n = clean.shape
        per = max(1, min(b, (128 << 20) // max(1, 2 * n * clean.element_size())))
        lens = None if lengths is None else torch.as_tensor(lengths).to(torch.int32).reshape(-1)
        cur = torch.cuda.current_stream(self.device)
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(self.device)
        copy = self._copy_stream
        copy.wait_stream(cur)
        outs = []
        staged = None
        starts = list(range(0, b, per))

        def upload(i0):
            with torch.cuda.stream(copy):
                c = clean[i0:i0 + per].to(self.device, non_blocking=True)
                d = deg[i0:i0 + per].to(self.device, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy)
            return c, d, ev

        staged = upload(starts[0])
        for k, i0 in enumerate(starts):
            c, d, ev = staged
            if k + 1 < len(starts):
                staged = upload(starts[k + 1])          # in flight while this chunk is scored
            cur.wait_event(ev)
            c.record_stream(cur)
            d.record_stream(cur)
            outs.append(self.score_tensors(c, d, None if lens is None else lens[i0:i0 + per]))
        return torch.cat(outs).cpu()

    # ------------------------------------------------------------------ helpers
    def _get_workspace(self, nbytes: int) -> torch.Tensor:
        if self._workspace is None or self._workspace.numel() < nbytes or self._workspace.device != self.device:
            self._workspace = None
            self._workspace = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=self.device)
        return self._workspace

    @staticmethod
    def _lengths_tensor(lengths, batch: int, n: int, device) -> torch.Tensor | None:
        if lengths is None:
            return None
        t = torch.as_tensor(lengths).to(torch.int32).reshape(-1)
        if t.numel() != batch:
            raise Exception("`lengths` must have one entry per batch item")
        if t.numel() and (int(t.min()) < 0 or int(t.max()) > n):
            raise Exception("`lengths` entries must lie in [0, samples]")
        return t.to(device).contiguous()
