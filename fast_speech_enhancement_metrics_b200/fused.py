"""PESQ + STOI/ESTOI on ONE host->device upload.

Callers of the reference always score both metrics on the same pair of tensors
(README.md:29-30, benchmark_metrics.py:22,24).  With host tensors the PCIe copy dominates the
end-to-end time, so `score_pesq_stoi` hands the pair to the library once: every chunk is copied
once and both kernel pipelines run on it (SURVEY.md 8f, rank 1).  Results are identical to
calling the two metric objects separately.  (Round 1's single-READ first-pass kernel and two-stream
overlap modes measured slower than the two separate first kernels on B200 and were removed; DESIGN.md.)
"""
from __future__ import annotations

import ctypes as C
import warnings

import torch

from . import _lib
from .base import check_score, make_batch, score_host, stream_ptr
from .PESQ import PESQ
from .STOI import STOI


def score_pesq_stoi_tensors(pesq: PESQ, stoi: STOI, clean: torch.Tensor, deg: torch.Tensor, lengths=None):
    """Device-resident scoring of both metrics: [B, n] float32 / int16 / float16 CUDA tensors -> (scores[3, B] f32 = PESQ / STOI /
    ESTOI rows, pesq_status[B], kept_frames[B], stoi_status[B]) CUDA tensors; stream-ordered, no host sync
    (C ABI fsem_pesq_stoi_score_f32: the two kernel chains back to back on the current stream)."""
    clean, deg = pesq._on_device(clean), pesq._on_device(deg)
    if stoi.device != pesq.device:
        raise Exception("both metrics must live on the same CUDA device")
    b, n = clean.shape
    lens = pesq._lengths_tensor(lengths, b, n, clean.device)
    scores = torch.empty(3, b, dtype=torch.float32, device=clean.device)
    pst = torch.empty(b, dtype=torch.int32, device=clean.device)
    kept = torch.empty(b, dtype=torch.int32, device=clean.device)
    sst = torch.empty(b, dtype=torch.int32, device=clean.device)
    batch, clean, deg = make_batch(clean, deg, lens)
    with torch.cuda.device(clean.device):
        wp = pesq._get_workspace(pesq._lib.fsem_pesq_workspace_bytes(pesq._ctx, b, n))
        wsb = stoi._get_workspace(stoi._lib.fsem_stoi_workspace_bytes(stoi._ctx, b, n))
        check_score(pesq._lib.fsem_pesq_stoi_score(
            pesq._ctx, stoi._ctx, C.byref(batch), _lib.dtype_code(clean.dtype), scores[0].data_ptr(), pst.data_ptr(), scores[1].data_ptr(),
            scores[2].data_ptr(), kept.data_ptr(), sst.data_ptr(), wp.data_ptr(), wp.numel(), wsb.data_ptr(),
            wsb.numel(), stream_ptr(clean.device)))
    pesq._last_shape = (b, n)
    stoi._last_shape = (b, n)
    stoi._last_lengths = lens
    return scores, pst, kept, sst


def score_pesq_stoi(pesq: PESQ, stoi: STOI, clean_speech: torch.Tensor, denoised_speech: torch.Tensor,
                    lengths=None) -> list[dict[str, float]]:
    """Returns [{"PESQ": ..., "STOI": ..., "ESTOI": ...}, ...], one dict per batch row.
    `stoi` must have been built for the tensors' sample rate (e.g. STOI(16000)) and `pesq` for 16 kHz."""
    if stoi.sample_rate != pesq.sample_rate:
        raise Exception("both metrics must be built for the sample rate of the audio")
    clean, deg = pesq.prepare_inputs(clean_speech, denoised_speech)
    assert clean is not None
    if clean.is_cuda:
        # device-resident tensors: one library call for both kernel chains
        scores, pst, kept, _ = score_pesq_stoi_tensors(pesq, stoi, clean, deg, lengths)
        packed = torch.cat([scores, pst.to(torch.float32)[None], kept.to(torch.float32)[None]]).cpu()
        mos, sc, pst, kept = packed[0], packed[1:3], packed[3].to(torch.int32), packed[4].to(torch.int32)
    else:
        mos, pst, sc, kept, _ = score_host(pesq, stoi, clean, deg, lengths)
    if lengths is not None and bool((pst == _lib.ITEM_TOO_SHORT).any()):
        raise RuntimeError("PESQ needs at least 20 frames of 512/256 samples for every item")
    stoi.last_kept_frames = kept
    if int(kept.max()) <= stoi.N + 1:
        warnings.warn("Not enough non-silent frames. Please check your sound files", RuntimeWarning, stacklevel=2)
        raise TypeError("iteration over a 0-d tensor")
    return [{"PESQ": p, "STOI": s, "ESTOI": e} for p, s, e in zip(mos.tolist(), sc[0].tolist(), sc[1].tolist())]


class CapturedScorer:
    """PESQ and/or STOI/ESTOI of FIXED device buffers as ONE CUDA graph (C ABI fsem_graph_*).

    The two kernel chains share nothing but their read-only inputs, so the graph runs them as parallel branches
    (and, for large batches, one pair of branches per slice of the batch: the tail of every kernel overlaps with
    another branch's work): a replay costs one graph launch and the longer chain instead of 3 + 7 launches back to
    back.  This is the path for the small batches of the reference's README example (4 x 10 s, README.md:21-30),
    where every kernel sits on its latency floor, and for scoring inside a loop that refills the same buffers
    (validation steps).  `slices` = parts the batch is cut into (0: the library's choice); the scores do not depend
    on it.  Static-buffer contract of CUDA graphs: `clean` / `deg` (and `lengths`) are captured BY ADDRESS -- write
    the next batch into them in place (`clean.copy_(...)`) and call the scorer again.  Results are bit-identical to
    `score_pesq_stoi_tensors` on the same buffers (same kernels, same launch shapes).

        scorer = CapturedScorer(PESQ(16000), STOI(16000), clean_cuda, deg_cuda)
        rows = scorer()                      # [{"PESQ": .., "STOI": .., "ESTOI": ..}, ...]
        clean_cuda.copy_(next_clean); deg_cuda.copy_(next_deg); rows = scorer()
    """

    def __init__(self, pesq: PESQ | None, stoi: STOI | None, clean: torch.Tensor, deg: torch.Tensor, lengths=None,
                 slices: int = 0):
        if pesq is None and stoi is None:
            raise Exception("CapturedScorer needs at least one metric")
        owner = pesq if pesq is not None else stoi
        if pesq is not None and stoi is not None:
            if stoi.device != pesq.device:
                raise Exception("both metrics must live on the same CUDA device")
            if stoi.sample_rate != pesq.sample_rate:
                raise Exception("both metrics must be built for the sample rate of the audio")
        if not (clean.is_cuda and deg.is_cuda) or clean.device != owner.device:
            raise Exception("CapturedScorer captures device buffers on the metric's device (got %s)" % clean.device)
        ptrs = (clean.data_ptr(), deg.data_ptr())
        clean, deg = owner.prepare_inputs(clean, deg)
        if (clean.data_ptr(), deg.data_ptr()) != ptrs:
            raise Exception("CapturedScorer captures buffers in place: rows must have unit stride along time")
        b, n = clean.shape
        if deg.stride(0) != clean.stride(0) and b > 1:
            raise Exception("`clean_speech` and `denoised_speech` need the same row pitch to be captured in place")
        self.pesq, self.stoi, self.clean, self.deg = pesq, stoi, clean, deg
        self._lib = owner._lib
        self.device = owner.device
        self.lengths = owner._lengths_tensor(lengths, b, n, clean.device)
        self.scores = torch.full((3, b), float("nan"), dtype=torch.float32, device=clean.device)
        self.pesq_status = torch.zeros(b, dtype=torch.int32, device=clean.device)
        self.kept_frames = torch.zeros(b, dtype=torch.int32, device=clean.device)
        self.stoi_status = torch.zeros(b, dtype=torch.int32, device=clean.device)
        # the library cuts the batch into `slices` parts (0: its own choice) and owns the graph's workspaces
        self._handle = C.c_void_p()
        batch, _, _ = make_batch(clean, deg, self.lengths)      # same pitch (checked above): points at clean / deg
        with torch.cuda.device(self.device):
            check_score(self._lib.fsem_graph_create(
                C.byref(self._handle), pesq._ctx if pesq is not None else None, stoi._ctx if stoi is not None else None,
                C.byref(batch), _lib.dtype_code(clean.dtype), self.scores[0].data_ptr(), self.pesq_status.data_ptr(),
                self.scores[1].data_ptr(), self.scores[2].data_ptr(), self.kept_frames.data_ptr(),
                self.stoi_status.data_ptr(), int(slices)))
        self.slices = int(self._lib.fsem_graph_slices(self._handle))
        self.kernel_nodes = int(self._lib.fsem_graph_nodes(self._handle))

    def replay(self):
        """One graph launch on the current stream; returns the captured output tensors (scores[3, B] = PESQ / STOI /
        ESTOI rows, pesq_status, kept_frames, stoi_status), valid in stream order, overwritten by the next replay."""
        if not getattr(self, "_handle", None):
            raise Exception("CapturedScorer is closed")
        with torch.cuda.device(self.device):
            _lib.check(self._lib.fsem_graph_launch(self._handle, stream_ptr(self.device)))
        return self.scores, self.pesq_status, self.kept_frames, self.stoi_status

    def __call__(self) -> list[dict[str, float]]:
        scores, pst, kept, _ = self.replay()
        packed = torch.cat([scores, pst.to(torch.float32)[None], kept.to(torch.float32)[None]]).cpu()   # one D2H copy
        if self.pesq is not None and self.lengths is not None and bool((packed[3] == _lib.ITEM_TOO_SHORT).any()):
            raise RuntimeError("PESQ needs at least 20 frames of 512/256 samples for every item")
        if self.stoi is not None:
            self.stoi.last_kept_frames = packed[4].to(torch.int32)
            if int(packed[4].max()) <= self.stoi.N + 1:
                warnings.warn("Not enough non-silent frames. Please check your sound files", RuntimeWarning, stacklevel=2)
                raise TypeError("iteration over a 0-d tensor")
        names = ([("PESQ", 0)] if self.pesq is not None else []) + ([("STOI", 1), ("ESTOI", 2)] if self.stoi is not None else [])
        cols = {k: packed[i].tolist() for k, i in names}
        return [{k: cols[k][j] for k, _ in names} for j in range(packed.shape[1])]

    def close(self):
        h, self._handle = getattr(self, "_handle", None), C.c_void_p()   # a constructor that raised never set it
        if h:
            try:
                torch.cuda.synchronize(self.device)
                self._lib.fsem_graph_destroy(h)
            except Exception:
                pass

    def __del__(self):
        self.close()
