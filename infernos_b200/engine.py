"""Python face of the B200 TTS tail: owns one C-ABI context per GPU and exposes the three callables the
reference engine holds (vocoder / chunker / resampler: /root/reference/HelloSippyTTSRT/HelloSippyRTPipe.py:236,237,240)
plus the fused tail.  torch is used only for device memory and streams."""
from __future__ import annotations

import ctypes
import operator
from typing import Dict, Optional, Sequence, Tuple

import torch

from . import _lib, resample_taps
from ._lib import LAW_ALAW, LAW_NONE, LAW_ULAW, MODE_BF16, MODE_FP32, TAIL_APPLY_POSTNET

_MODES = {"fp32": MODE_FP32, "bf16": MODE_BF16, MODE_FP32: MODE_FP32, MODE_BF16: MODE_BF16}
_taps_set = set()


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _require_cuda(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"{name} must live on a CUDA device (infernos_b200 has no CPU path)")
    if t.dtype != dtype:
        raise RuntimeError(f"{name} must be {dtype}, got {t.dtype}")
    return t.contiguous()


def ensure_taps(device: torch.device) -> None:
    """Hands torchaudio-identical taps to the library once per device (it also has them built in)."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx in _taps_set:
        return
    lib = _lib.load()
    d = resample_taps.down_taps().numpy()
    u = resample_taps.up_taps().reshape(30).numpy()
    with torch.cuda.device(idx):
        _lib.check(lib.b2_set_resample_taps(d.ctypes.data_as(ctypes.c_void_p), u.ctypes.data_as(ctypes.c_void_p)), "set_resample_taps")
    _taps_set.add(idx)


class TTSTail:
    """One context = packed weights + workspaces + the pre_frames pool of the sessions on one GPU."""

    def __init__(self, device, vocoder_sd: Dict[str, torch.Tensor], chunker_sd: Optional[Dict[str, torch.Tensor]] = None,
                 mode="bf16", max_sessions: int = 1024, max_windows: int = 1024,
                 postnet_sd: Optional[Dict[str, torch.Tensor]] = None):
        """postnet_sd (optional, SURVEY section 8 f3): state_dict of transformers SpeechT5SpeechDecoderPostnet (or of the whole
        SpeechT5ForTextToSpeech / its `speech_decoder_postnet`): only the `layers.*` conv / batch-norm tensors are taken."""
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("infernos_b200 runs on CUDA devices only (no CPU fallback)")
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device is visible (infernos_b200 has no CPU fallback)")
        self.index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", self.index)
        self.mode = _MODES[mode]
        self.max_sessions, self.max_windows = int(max_sessions), int(max_windows)
        self.ctx = self.lib.b2_ctx_create(self.index, self.mode, self.max_sessions, self.max_windows)
        if not self.ctx:
            raise RuntimeError("b2_ctx_create: " + self.lib.b2_last_error(None).decode())
        try:
            self._load(vocoder_sd, self.lib.b2_load_vocoder_tensor)
            if chunker_sd is not None:
                self._load(chunker_sd, self.lib.b2_load_chunker_tensor)
            if postnet_sd is not None:
                self._load(postnet_layers(postnet_sd), self.lib.b2_load_postnet_tensor)
            _lib.check(self.lib.b2_weights_finalize(self.ctx), "weights_finalize")
            ensure_taps(self.device)
        except Exception:
            self.close()
            raise
        self.has_chunker = chunker_sd is not None
        self.has_postnet = postnet_sd is not None

    def _load(self, sd, fn):
        for k, v in sd.items():
            t = v.detach().to("cpu", torch.float32).contiguous()
            shape = (ctypes.c_int64 * t.dim())(*t.shape)
            _lib.check(fn(self.ctx, k.encode(), ctypes.c_void_p(t.data_ptr()), shape, t.dim()), f"load {k}")

    def close(self):
        for sch in list(getattr(self, "_schedulers", ())):      # a serving loop's threads use this context: stop them first
            sch.close()
        if getattr(self, "ctx", None):
            self.lib.b2_ctx_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def device_bytes(self) -> int:
        return int(self.lib.b2_ctx_device_bytes(self.ctx))

    # ---- the reference's three callables ------------------------------------------------------------
    def vocoder(self, spectrogram: torch.Tensor) -> torch.Tensor:
        """SpeechT5HifiGan.forward: (W,T,80) -> (W,256*T); un-batched (T,80) -> (256*T,)."""
        squeeze = spectrogram.dim() == 2
        x = spectrogram.unsqueeze(0) if squeeze else spectrogram
        in_dtype = x.dtype
        x = _require_cuda(x.to(torch.float32), torch.float32, "spectrogram")
        W, T, nm = x.shape
        if nm != 80:
            raise RuntimeError(f"spectrogram must have 80 mel bins, got {nm}")
        out = torch.empty(W, T * 256, device=x.device, dtype=torch.float32)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_vocoder_forward(self.ctx, x.data_ptr(), W, T, out.data_ptr(), _stream_ptr(x.device)), "vocoder_forward")
        out = out.to(in_dtype) if in_dtype != torch.float32 else out
        return out.squeeze(0) if squeeze else out

    def chunker(self, mel: torch.Tensor, audio: torch.Tensor) -> torch.Tensor:
        """AmendmentNetwork1.forward: mel (W,12,80), audio (W,3072) -> (W,2048)."""
        in_dtype = audio.dtype
        m = _require_cuda(mel.to(torch.float32), torch.float32, "mel")
        a = _require_cuda(audio.to(torch.float32), torch.float32, "audio")
        W = a.size(0)
        if tuple(m.shape) != (W, 12, 80) or a.size(1) != 3072:
            raise RuntimeError(f"chunker expects mel (W,12,80) and audio (W,3072), got {tuple(m.shape)} and {tuple(a.shape)}")
        out = torch.empty(W, 2048, device=a.device, dtype=torch.float32)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_chunker_forward(self.ctx, m.data_ptr(), a.data_ptr(), W, out.data_ptr(), _stream_ptr(a.device)), "chunker_forward")
        return out.to(in_dtype) if in_dtype != torch.float32 else out

    def resampler(self, audio: torch.Tensor) -> torch.Tensor:
        """torchaudio Resample(16000, 8000): (..., L) -> (..., ceil(L/2))."""
        return resample_2to1(audio)

    def postnet(self, spectrogram: torch.Tensor) -> torch.Tensor:
        """SpeechT5SpeechDecoderPostnet.postnet (the call at HelloSippyRTPipe.py:230): (B,T,80) -> (B,T,80)."""
        if not self.has_postnet:
            raise RuntimeError("this TTSTail was built without post-net weights (postnet_sd)")
        in_dtype = spectrogram.dtype
        x = _require_cuda(spectrogram.to(torch.float32), torch.float32, "spectrogram")
        B, T, nm = x.shape
        if nm != 80:
            raise RuntimeError(f"spectrogram must have 80 mel bins, got {nm}")
        out = torch.empty_like(x)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_postnet_forward(self.ctx, x.data_ptr(), B, T, out.data_ptr(), _stream_ptr(x.device)), "postnet_forward")
        return out.to(in_dtype) if in_dtype != torch.float32 else out

    # ---- fused tail ----------------------------------------------------------------------------------
    def tail(self, slots: torch.Tensor, mel: torch.Tensor, law: int = LAW_ULAW, want_g711: bool = True,
             want_audio: bool = True, apply_postnet: bool = False) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
        """slots (B,) int32 cuda, mel (B,n,80) fp32 cuda -> (g711 (B,n*128) uint8 | None, audio8k (B,n*128) fp32 | None).
        apply_postnet: mel holds the frames BEFORE the post-net (feat_out's output); the post-net runs in the same call."""
        s = _require_cuda(slots, torch.int32, "slots")
        m = _require_cuda(mel, torch.float32, "mel")
        B, n, nm = m.shape
        if nm != 80 or s.numel() != B:
            raise RuntimeError("tail expects mel (B,n,80) and slots (B,)")
        g = torch.empty(B, n * 128, device=m.device, dtype=torch.uint8) if want_g711 else None
        a = torch.empty(B, n * 128, device=m.device, dtype=torch.float32) if want_audio else None
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_tts_tail2(self.ctx, s.data_ptr(), m.data_ptr(), B, n, law if want_g711 else LAW_NONE,
                                             TAIL_APPLY_POSTNET if apply_postnet else 0,
                                             g.data_ptr() if g is not None else None, a.data_ptr() if a is not None else None,
                                             _stream_ptr(m.device)), "tts_tail")
        return g, a

    def tail_host(self, slots: torch.Tensor, mel: torch.Tensor, out_g711: Optional[torch.Tensor], out_audio: Optional[torch.Tensor] = None,
                  law: int = LAW_ULAW, apply_postnet: bool = False) -> None:
        """End-to-end entry with HOST (ideally pinned) tensors; returns after the outputs are in host memory."""
        if slots.is_cuda or mel.is_cuda:
            raise RuntimeError("tail_host takes host tensors")
        B, n, _ = mel.shape
        assert slots.dtype == torch.int32 and mel.dtype == torch.float32 and slots.is_contiguous() and mel.is_contiguous()
        if out_g711 is not None:
            assert out_g711.dtype == torch.uint8 and out_g711.numel() == B * n * 128 and out_g711.is_contiguous()
        if out_audio is not None:
            assert out_audio.dtype == torch.float32 and out_audio.numel() == B * n * 128 and out_audio.is_contiguous()
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_tts_tail_host2(self.ctx, slots.data_ptr(), mel.data_ptr(), B, n, law,
                                                 TAIL_APPLY_POSTNET if apply_postnet else 0,
                                                 out_g711.data_ptr() if out_g711 is not None else None,
                                                 out_audio.data_ptr() if out_audio is not None else None,
                                                 _stream_ptr(self.device)), "tts_tail_host")

    def poll_errors(self) -> None:
        """Synchronises the current stream and raises if an earlier asynchronous tail call was handed a slot id outside the pool or
        twice in one call (the device-side check of k_build_windows)."""
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_ctx_poll_errors(self.ctx, _stream_ptr(self.device)), "poll_errors")

    TAP_NAMES = ("conv_pre", "up0", "stage0", "up1", "stage1", "up2", "stage2", "up3", "stage3")
    TAP_CH = (512, 256, 256, 128, 128, 64, 64, 32, 32)
    TAP_UP = (1, 4, 4, 16, 16, 64, 64, 256, 256)

    def vocoder_with_taps(self, spectrogram: torch.Tensor, names: Sequence[str] = TAP_NAMES):
        """vocoder() plus the fp32 stage-boundary tensors of modeling_speecht5.py:3062-3072, returned channel-FIRST (W, C, T_stage)
        like the torch module's own intermediates (the library keeps them channels-last).  Parity-test hook (BASELINE config 2)."""
        x = _require_cuda(spectrogram.to(torch.float32), torch.float32, "spectrogram")
        W, T, _ = x.shape
        if W * T > 12 * self.max_windows:
            raise RuntimeError("vocoder_with_taps: the call must fit one sub-batch (W*T <= 12*max_windows)")
        bufs, ptrs = {}, (ctypes.c_void_p * 9)()
        for i, n in enumerate(self.TAP_NAMES):
            if n in names:
                bufs[n] = torch.empty(W, T * self.TAP_UP[i], self.TAP_CH[i], device=x.device, dtype=torch.float32)
                ptrs[i] = bufs[n].data_ptr()
        _lib.check(self.lib.b2_debug_set_taps(self.ctx, ptrs), "debug_set_taps")
        try:
            audio = self.vocoder(x)
        finally:
            _lib.check(self.lib.b2_debug_set_taps(self.ctx, None), "debug_set_taps")
        return audio, {n: b.transpose(1, 2) for n, b in bufs.items()}

    def profile_begin(self) -> None:
        _lib.check(self.lib.b2_profile_begin(self.ctx), "profile_begin")

    def profile_end(self):
        """-> ({class: ms}, {class: launches}) for classes conv_tc (per-layer tcgen05 convs), conv_f32, conv_post, resample_g711,
        other, resblock_tc (the fused tcgen05 ResBlock kernel)."""
        ms = (ctypes.c_double * 8)()
        n = (ctypes.c_uint64 * 8)()
        _lib.check(self.lib.b2_profile_end(self.ctx, ms, n), "profile_end")
        names = ["conv_tc", "conv_f32", "conv_post", "resample_g711", "other", "resblock_tc"]
        return {k: ms[i] for i, k in enumerate(names)}, {k: int(n[i]) for i, k in enumerate(names)}

    def reset_sessions(self, slots: Sequence[int]) -> None:
        arr = (ctypes.c_int32 * len(slots))(*[int(s) for s in slots])
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_session_reset(self.ctx, arr, len(slots), _stream_ptr(self.device)), "session_reset")

    def get_pre_frames(self, slot: int) -> torch.Tensor:
        out = torch.empty(4, 80, dtype=torch.float32)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_session_get_pre_frames(self.ctx, int(slot), out.data_ptr(), _stream_ptr(self.device)), "get_pre_frames")
        return out

    def set_pre_frames(self, slot: int, frames: torch.Tensor) -> None:
        f = frames.detach().to("cpu", torch.float32).contiguous()
        assert tuple(f.shape) == (4, 80)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_session_set_pre_frames(self.ctx, int(slot), f.data_ptr(), _stream_ptr(self.device)), "set_pre_frames")


class _Completion(ctypes.Structure):
    _fields_ = [("tag", ctypes.c_uint64), ("t_enqueue_ns", ctypes.c_int64), ("t_launch_ns", ctypes.c_int64), ("t_done_ns", ctypes.c_int64),
                ("g711_offset", ctypes.c_int64), ("slot", ctypes.c_int32), ("nbytes", ctypes.c_int32), ("batch_sessions", ctypes.c_int32),
                ("reserved_", ctypes.c_int32)]


class _SchedStats(ctypes.Structure):
    _fields_ = [(k, ctypes.c_uint64) for k in ("sub_batches", "sessions", "padded_sessions", "graph_launches", "graphs_built", "max_sub_batch",
                                               "capacity", "depth")]


class TailScheduler:
    """Latency-bounded serving loop over one TTSTail (include/infernos_b200.h, b2_sched_*): submit (slot, mel chunk) pairs from any
    thread; sub-batches are formed adaptively and run as H2D -> one CUDA-graph launch -> D2H with `depth` of them in flight.
    While a scheduler exists it owns the tail's workspaces: do not call tail.tail()/vocoder() concurrently."""

    def __init__(self, tail: "TTSTail", nframes: int = 8, law: int = LAW_ULAW, apply_postnet: bool = False, max_batch: int = 0,
                 depth: int = 2, use_graphs: bool = True, poll_capacity: int = 4096):
        self.tail, self.lib, self.nframes = tail, tail.lib, int(nframes)
        with torch.cuda.device(tail.index):
            self.h = self.lib.b2_sched_create(tail.ctx, self.nframes, law, TAIL_APPLY_POSTNET if apply_postnet else 0, int(max_batch), int(depth),
                                              1 if use_graphs else 0)
        if not self.h:
            raise RuntimeError("b2_sched_create: " + self.lib.b2_last_error(None).decode())
        if not hasattr(tail, "_schedulers"):
            tail._schedulers = []
        tail._schedulers.append(self)
        self._cap = int(poll_capacity)
        self._recs = (_Completion * self._cap)()
        self._bytes = torch.empty(self._cap * self.nframes * 128, dtype=torch.uint8)

    def close(self):
        if getattr(self, "h", None):
            self.lib.b2_sched_destroy(self.h)
            self.h = None
            if self in getattr(self.tail, "_schedulers", []):
                self.tail._schedulers.remove(self)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_policy(self, min_batch: int = 0, max_wait_us: int = 0) -> None:
        _lib.check(self.lib.b2_sched_set_policy(self.h, int(min_batch), int(max_wait_us)), "sched_set_policy")

    def submit(self, slots: torch.Tensor, mel: torch.Tensor, t_enqueue_ns: Optional[torch.Tensor] = None, tags: Optional[torch.Tensor] = None) -> None:
        """slots (n,) int32, mel (n, nframes, 80) fp32, both on the HOST (any memory; they are copied into pinned staging);
        t_enqueue_ns (n,) int64 CLOCK_MONOTONIC arrival stamps (default: now); tags (n,) uint64 (default: the slot id)."""
        n = slots.numel()
        assert not slots.is_cuda and not mel.is_cuda and slots.dtype == torch.int32 and mel.dtype == torch.float32
        assert slots.is_contiguous() and mel.is_contiguous() and mel.numel() == n * self.nframes * 80
        te = t_enqueue_ns.data_ptr() if t_enqueue_ns is not None else None
        tg = tags.data_ptr() if tags is not None else None
        if t_enqueue_ns is not None:
            assert t_enqueue_ns.dtype == torch.int64 and t_enqueue_ns.numel() == n and t_enqueue_ns.is_contiguous()
        if tags is not None:
            assert tags.dtype in (torch.int64, torch.uint64) and tags.numel() == n and tags.is_contiguous()
        _lib.check(self.lib.b2_sched_submit(self.h, slots.data_ptr(), mel.data_ptr(), n, te, tg), "sched_submit")

    def poll(self, timeout_ms: int = 0, want_bytes: bool = True):
        """-> (records, bytes): records is a ctypes array slice of finished chunks (tag, slot, t_enqueue_ns, t_launch_ns, t_done_ns,
        batch_sessions, g711_offset), bytes the uint8 tensor their offsets point into (valid until the next poll)."""
        n = self.lib.b2_sched_poll(self.h, self._recs, self._cap, self._bytes.data_ptr() if want_bytes else None, self._bytes.numel(), int(timeout_ms))
        if n < 0:
            raise RuntimeError("infernos_b200 sched_poll: " + self.lib.b2_last_error(None).decode())
        return self._recs[:n], self._bytes

    def flush(self, timeout_ms: int = 60000) -> None:
        _lib.check(self.lib.b2_sched_flush(self.h, int(timeout_ms)), "sched_flush")

    def prebuild(self, max_sessions: int = 0) -> None:
        """Build the CUDA graphs of every sub-batch bucket up to `max_sessions` (0: up to max_batch) now, while the scheduler is idle, instead of
        on the serving path the first time a sub-batch of that size turns up."""
        _lib.check(self.lib.b2_sched_prebuild(self.h, int(max_sessions)), "sched_prebuild")

    def stats(self) -> dict:
        st = _SchedStats()
        _lib.check(self.lib.b2_sched_get_stats(self.h, ctypes.byref(st)), "sched_get_stats")
        return {k: int(getattr(st, k)) for k, _ in _SchedStats._fields_}


def decoder_position_table(max_len: int, dim: int = 768) -> torch.Tensor:
    """SpeechT5ScaledPositionalEncoding.pe (transformers modeling_speecht5.py:405-412), computed with the same torch expressions so that
    the table the library adds is bit-identical to the module's buffer."""
    import math
    pe = torch.zeros(max_len, dim)
    position = torch.arange(0, max_len).unsqueeze(1)
    div_term = torch.exp(torch.arange(0, dim, 2, dtype=torch.int64).float() * -(math.log(10000.0) / dim))
    pe[:, 0::2] = torch.sin(position.float() * div_term)
    pe[:, 1::2] = torch.cos(position.float() * div_term)
    return pe


class TTSDecoder:
    """The autoregressive SpeechT5 speech decoder on the GPU (b2_dec_*, SURVEY section 8 f3): prenet -> six decoder layers with a slot KV
    cache -> feat_out / prob_out, the front half of the reference's infer() (HelloSippyRTPipe.py:195-229).  `sd` is a state_dict that
    holds the `speecht5.decoder.*` and `speech_decoder_postnet.{feat_out,prob_out}.*` tensors of transformers SpeechT5ForTextToSpeech
    (the whole model's state_dict will do)."""

    def __init__(self, device, sd: Dict[str, torch.Tensor], mode="bf16", max_sessions: int = 64, max_rows: int = 0, max_steps: int = 512,
                 max_enc_len: int = 128):
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda" or not torch.cuda.is_available():
            raise RuntimeError("infernos_b200 runs on CUDA devices only (no CPU fallback)")
        self.index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", self.index)
        self.mode = _MODES[mode]
        self.max_sessions, self.max_steps, self.max_enc_len = int(max_sessions), int(max_steps), int(max_enc_len)
        self.max_rows = int(max_rows) if max_rows else min(self.max_sessions, 1024)
        self.h = self.lib.b2_dec_create(self.index, self.mode, self.max_sessions, self.max_rows, self.max_steps, self.max_enc_len)
        if not self.h:
            raise RuntimeError("b2_dec_create: " + self.lib.b2_last_error(None).decode())
        try:
            n = 0
            for k, v in sd.items():
                if not (k.startswith("speecht5.decoder.prenet.") or k.startswith("speecht5.decoder.wrapped_decoder.") or
                        k.startswith("speech_decoder_postnet.feat_out.") or k.startswith("speech_decoder_postnet.prob_out.")):
                    continue
                if k.endswith("encode_positions.pe"):
                    continue
                self._load(k, v)
                n += 1
            if n != 8 + 1 + 6 * 26 + 4:
                raise RuntimeError(f"decoder state_dict: expected {8 + 1 + 6 * 26 + 4} tensors, found {n}")
            self._load("pe", decoder_position_table(self.max_steps))
            with torch.cuda.device(self.index):
                _lib.check(self.lib.b2_dec_finalize(self.h), "dec_finalize")
        except Exception:
            self.close()
            raise

    def _load(self, k, v):
        t = v.detach().to("cpu", torch.float32).contiguous()
        shape = (ctypes.c_int64 * max(1, t.dim()))(*t.shape)
        _lib.check(self.lib.b2_dec_load_tensor(self.h, k.encode(), ctypes.c_void_p(t.data_ptr()), shape, t.dim()), f"dec load {k}")

    def close(self):
        if getattr(self, "h", None):
            self.lib.b2_dec_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def device_bytes(self) -> int:
        return int(self.lib.b2_dec_device_bytes(self.h))

    def start(self, slots: torch.Tensor, enc: torch.Tensor, enc_len: Optional[torch.Tensor], speaker: torch.Tensor) -> None:
        """New sentences: slots (n,) int32 cuda, enc (n, L, 768) = encoder_last_hidden_state, enc_len (n,) int32 valid prefix lengths (or
        None), speaker (n, 512)."""
        s = _require_cuda(slots, torch.int32, "slots")
        e = _require_cuda(enc.to(torch.float32), torch.float32, "enc")
        sp = _require_cuda(speaker.to(torch.float32), torch.float32, "speaker")
        n, L, hdim = e.shape
        if hdim != 768 or tuple(sp.shape) != (n, 512) or s.numel() != n:
            raise RuntimeError("decoder.start expects enc (n, L, 768), speaker (n, 512), slots (n,)")
        el = _require_cuda(enc_len, torch.int32, "enc_len") if enc_len is not None else None
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_dec_start(self.h, s.data_ptr(), e.data_ptr(), el.data_ptr() if el is not None else None, sp.data_ptr(), n, L,
                                             _stream_ptr(self.device)), "dec_start")

    def steps(self, slots: torch.Tensor, nsteps: int = 16, masks: Optional[torch.Tensor] = None, seed: int = 0):
        """-> (mel (n, 2*nsteps, 80) fp32 cuda: feat_out's frames, BEFORE the post-net; prob (n, nsteps, 2) fp32 cuda)."""
        s = _require_cuda(slots, torch.int32, "slots")
        n = s.numel()
        mel = torch.empty(n, 2 * nsteps, 80, device=self.device, dtype=torch.float32)
        prob = torch.empty(n, nsteps, 2, device=self.device, dtype=torch.float32)
        mk = None
        if masks is not None:
            mk = _require_cuda(masks.to(torch.float32), torch.float32, "masks")
            if tuple(mk.shape) != (nsteps, 2, 256):
                raise RuntimeError("masks must be (nsteps, 2, 256)")
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_dec_steps(self.h, s.data_ptr(), n, int(nsteps), mk.data_ptr() if mk is not None else None, int(seed) & (2 ** 64 - 1),
                                             mel.data_ptr(), prob.data_ptr(), _stream_ptr(self.device)), "dec_steps")
        return mel, prob

    def set_graphs(self, on: bool) -> None:
        _lib.check(self.lib.b2_dec_set_graphs(self.h, 1 if on else 0), "dec_set_graphs")

    def poll_errors(self) -> None:
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_dec_poll_errors(self.h, _stream_ptr(self.device)), "dec_poll_errors")

    def get_step(self, slot: int) -> int:
        v = ctypes.c_int32(0)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_dec_get_step(self.h, int(slot), ctypes.byref(v), _stream_ptr(self.device)), "dec_get_step")
        return int(v.value)


ENCODER_TENSORS = 2 + 2 + 1 + 12 * 16       # prenet (embedding, alpha), first LayerNorm, pe_k, 12 layers x 16


class TTSEncoder:
    """The SpeechT5 text encoder on the GPU (b2_enc_*): token ids -> encoder_last_hidden_state, what the reference runs once per sentence
    (HelloSippyRTPipe.py:111-116).  `sd` is a state_dict that holds the `speecht5.encoder.*` tensors of transformers SpeechT5ForTextToSpeech
    (the whole model's state_dict will do).  Only the valid tokens of a batch are computed: sentences are packed back to back into passes
    of at most `max_tokens` rows; `max_len` (<= 450, the model's max_text_positions) bounds the padded length of a call."""

    def __init__(self, device, sd: Dict[str, torch.Tensor], mode="bf16", max_tokens: int = 16384, max_len: int = 450):
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda" or not torch.cuda.is_available():
            raise RuntimeError("infernos_b200 runs on CUDA devices only (no CPU fallback)")
        self.index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", self.index)
        self.mode = _MODES[mode]
        self.max_tokens, self.max_len = int(max_tokens), int(max_len)
        self.h = self.lib.b2_enc_create(self.index, self.mode, self.max_tokens, self.max_len)
        if not self.h:
            raise RuntimeError("b2_enc_create: " + self.lib.b2_last_error(None).decode())
        try:
            n = 0
            for k, v in sd.items():
                if not k.startswith("speecht5.encoder.") or k.endswith("encode_positions.pe"):
                    continue
                self._load(k, v)
                n += 1
            if n != ENCODER_TENSORS:
                raise RuntimeError(f"encoder state_dict: expected {ENCODER_TENSORS} tensors, found {n}")
            self._load("pe", decoder_position_table(self.max_len))
            with torch.cuda.device(self.index):
                _lib.check(self.lib.b2_enc_finalize(self.h), "enc_finalize")
        except Exception:
            self.close()
            raise

    def _load(self, k, v):
        t = v.detach().to("cpu", torch.float32).contiguous()
        shape = (ctypes.c_int64 * max(1, t.dim()))(*t.shape)
        _lib.check(self.lib.b2_enc_load_tensor(self.h, k.encode(), ctypes.c_void_p(t.data_ptr()), shape, t.dim()), f"enc load {k}")

    def close(self):
        if getattr(self, "h", None):
            self.lib.b2_enc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def device_bytes(self) -> int:
        return int(self.lib.b2_enc_device_bytes(self.h))

    def __call__(self, input_ids: torch.Tensor, attention_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        """input_ids (B, L) integer (host or device), attention_mask (B, L) 0/1 with every row a prefix of ones (right padding) or None ->
        (B, L, 768) fp32 on this device: encoder_last_hidden_state at valid positions, zeros at padded ones.  The `encoder` callable of
        B200Frontend."""
        if input_ids.dim() != 2:
            raise RuntimeError("input_ids must be (B, L)")
        B, L = input_ids.shape
        lens = None
        if attention_mask is not None:
            m = attention_mask.detach().to("cpu", torch.int32)
            if tuple(m.shape) != (B, L):
                raise RuntimeError(f"attention_mask {tuple(m.shape)} does not match input_ids {(B, L)}")
            lens = m.sum(1, dtype=torch.int32).contiguous()
            if not torch.equal(m, (torch.arange(L)[None] < lens[:, None]).to(torch.int32)):
                raise RuntimeError("attention_mask must be a prefix of ones in every row (right-padded sentences)")
        ids = input_ids.to(device=self.device, dtype=torch.int32).contiguous()
        out = torch.empty(B, L, 768, device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_enc_forward(self.h, ids.data_ptr(), lens.data_ptr() if lens is not None else None, B, L, out.data_ptr(),
                                               _stream_ptr(self.device)), "enc_forward")
        return out

    def poll_errors(self) -> None:
        """Synchronises the current stream and raises if an earlier call was given token ids outside [0, 81)."""
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b2_enc_poll_errors(self.h, _stream_ptr(self.device)), "enc_poll_errors")


class _TTSChunk(ctypes.Structure):
    _fields_ = [("tag", ctypes.c_uint64), ("call", ctypes.c_int64), ("admit_call", ctypes.c_int64), ("t_submit_ns", ctypes.c_int64),
                ("t_done_ns", ctypes.c_int64), ("g711_offset", ctypes.c_int64), ("nbytes", ctypes.c_int32), ("ended", ctypes.c_int32)]


class _TTSServerStats(ctypes.Structure):
    _fields_ = [(k, ctypes.c_uint64) for k in ("calls", "submitted", "admitted", "ended", "admission_rounds", "rows", "live_rows", "padded_rows",
                                               "graph_launches", "graphs_built", "max_rows", "capacity", "depth")]


class TTSServer:
    """Whole sentences in, G.711 chunks out (b2_tts_server_*): the reference's worker loop around infer() / unbatch_and_dispatch()
    (Cluster/InfernTTSWorker.py:83-92, HelloSippyRTPipe.py:195-259) as a native loop.  Every engine call admits the sentences submitted since
    the last one, runs 16 decoder steps over every live sentence whatever call admitted it, applies the stop rule on the GPU and runs the tail
    with the post-net; `depth` calls are in flight.  `tail` must hold post-net weights.  While the server exists it owns the tail, encoder
    and decoder handles: do not call them, and close the server before them (closing the tail closes it)."""

    def __init__(self, tail: "TTSTail", encoder: "TTSEncoder", decoder: "TTSDecoder", law: int = LAW_ULAW, depth: int = 2, threshold: float = 0.5,
                 minlenratio: float = 0.0, maxlenratio: float = 20.0, seed: int = 0, use_graphs: bool = True, poll_capacity: int = 4096):
        if law not in (LAW_ULAW, LAW_ALAW):
            raise RuntimeError(f"law must be LAW_ULAW or LAW_ALAW, got {law!r}")
        if not 1 <= int(depth) <= 4:
            raise RuntimeError(f"depth must be 1..4, got {depth!r}")
        if not tail.has_postnet:
            raise RuntimeError("TTSServer needs a TTSTail built with post-net weights (postnet_sd)")
        if not (minlenratio >= 0.0 and maxlenratio >= 0.0 and threshold == threshold):
            raise RuntimeError("threshold must be a number and minlenratio / maxlenratio >= 0")
        if int(poll_capacity) < 1:
            raise RuntimeError("poll_capacity must be >= 1")
        self.tail, self.encoder, self.decoder, self.lib = tail, encoder, decoder, tail.lib
        with torch.cuda.device(tail.index):
            self.h = self.lib.b2_tts_server_create(tail.ctx, encoder.h, decoder.h, int(law), int(depth), 1 if use_graphs else 0, float(threshold),
                                                   float(minlenratio), float(maxlenratio), int(seed) & (2 ** 64 - 1))
        if not self.h:
            raise RuntimeError("b2_tts_server_create: " + self.lib.b2_last_error(None).decode())
        if not hasattr(tail, "_schedulers"):
            tail._schedulers = []
        tail._schedulers.append(self)
        self._cap = int(poll_capacity)
        self._recs = (_TTSChunk * self._cap)()
        self._bytes = torch.empty(self._cap * 4096, dtype=torch.uint8)

    def close(self) -> None:
        """Stops the loop (work in flight is dropped) and frees the server; the tail, encoder and decoder stay usable."""
        if getattr(self, "h", None):
            self.lib.b2_tts_server_destroy(self.h)
            self.h = None
            if self in getattr(self.tail, "_schedulers", []):
                self.tail._schedulers.remove(self)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _handle(self):
        if not getattr(self, "h", None):
            raise RuntimeError("the TTSServer is closed")
        return self.h

    def submit(self, ids, speaker, tag: int) -> None:
        """One sentence: ids = token ids (a 1-D sequence or tensor of ints), speaker = (512,) or (1, 512) x-vector (normalised on the GPU),
        tag = the caller's unsigned 64-bit id, echoed in every record.  Blocks while every slot is busy."""
        self.submit_many([ids], [speaker], [tag])

    def submit_many(self, ids_list, speakers, tags) -> None:
        """Several sentences at once (lists of what submit() takes); when the slots allow, they are admitted in one round.  Nothing is
        enqueued if any of them is rejected."""
        if not (len(ids_list) == len(speakers) == len(tags)):
            raise RuntimeError("ids_list, speakers and tags must have the same length")
        n = len(ids_list)
        if n == 0:
            return
        toks, lens = [], []
        for ids in ids_list:
            t = torch.as_tensor(ids)
            if t.dim() == 2 and t.size(0) == 1:
                t = t[0]
            if t.numel() < 1:
                raise RuntimeError("a sentence needs at least one token")
            if t.dim() != 1 or t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
                raise RuntimeError("ids must be a 1-D sequence of integer token ids")
            if int(t.min()) < -2 ** 31 or int(t.max()) >= 2 ** 31:
                raise RuntimeError("token ids must fit in int32")
            toks.append(t.to("cpu", torch.int32))
            lens.append(t.numel())
        sp = []
        for s in speakers:
            v = torch.as_tensor(s).detach().to("cpu", torch.float32).reshape(-1)
            if v.numel() != 512:
                raise RuntimeError(f"a speaker vector must hold 512 values, got {v.numel()}")
            sp.append(v)
        tg = [int(t) for t in tags]
        if any(not 0 <= t < 2 ** 64 for t in tg):
            raise RuntimeError("tags must be unsigned 64-bit integers")
        h = self._handle()
        ids_t = torch.cat(toks).contiguous()
        lens_t = torch.tensor(lens, dtype=torch.int32)
        sp_t = torch.stack(sp).contiguous()
        tags_a = (ctypes.c_uint64 * n)(*tg)
        _lib.check(self.lib.b2_tts_server_submit(h, ids_t.data_ptr(), lens_t.data_ptr(), n, sp_t.data_ptr(), tags_a), "tts_server_submit")

    def cancel(self, tags) -> int:
        """Cancels every sentence submitted with one of `tags` (one unsigned 64-bit tag or a sequence of them) whose last record has not been
        made: the barge-in of TTSSndDispatch.cancel().  A pending sentence gets its last record at once (call -1, never admitted); an admitted
        one at the next engine call, unless a call already in flight ends it first.  Records of calls in flight still arrive with their bytes.
        A cancelled sentence's last record has nbytes 0 and `cancelled` True.  Returns the number of sentences found; unknown tags, sentences
        that have ended and repeated cancels count 0."""
        try:
            tg = [operator.index(tags)]
        except TypeError:
            try:
                tg = [operator.index(t) for t in tags]
            except TypeError:
                raise RuntimeError("tags must be unsigned 64-bit integers") from None
        if any(not 0 <= t < 2 ** 64 for t in tg):
            raise RuntimeError("tags must be unsigned 64-bit integers")
        h = self._handle()
        n = self.lib.b2_tts_server_cancel(h, (ctypes.c_uint64 * len(tg))(*tg), len(tg))
        if n < 0:
            raise RuntimeError("infernos_b200 tts_server_cancel: " + self.lib.b2_last_error(None).decode())
        return n

    def poll(self, timeout_ms: int = 0):
        """-> list of (record, bytes): record a dict with tag, call, admit_call, nbytes, ended, cancelled, t_submit_ns, t_done_ns; bytes the
        G.711 payload of that sentence in that call.  `ended` marks a sentence's last record; `cancelled` one that cancel() ended.
        timeout_ms: 0 = do not wait, < 0 = wait for the next completed call."""
        h = self._handle()
        n = self.lib.b2_tts_server_poll(h, self._recs, self._cap, self._bytes.data_ptr(), self._bytes.numel(), int(timeout_ms))
        if n < 0:
            raise RuntimeError("infernos_b200 tts_server_poll: " + self.lib.b2_last_error(None).decode())
        out = []
        raw = self._bytes.numpy()
        for r in self._recs[:n]:
            rec = {k: int(getattr(r, k)) for k, _ in _TTSChunk._fields_ if k != "g711_offset"}
            rec["cancelled"] = rec["ended"] == 2
            rec["ended"] = bool(rec["ended"])
            out.append((rec, raw[r.g711_offset:r.g711_offset + r.nbytes].tobytes()))
        return out

    def flush(self, timeout_ms: int = 600000) -> None:
        """Returns when every sentence submitted so far has ended (its records may still be waiting for poll)."""
        h = self._handle()
        _lib.check(self.lib.b2_tts_server_flush(h, int(timeout_ms)), "tts_server_flush")

    def stats(self) -> dict:
        h, st = self._handle(), _TTSServerStats()
        _lib.check(self.lib.b2_tts_server_get_stats(h, ctypes.byref(st)), "tts_server_get_stats")
        return {k: int(getattr(st, k)) for k, _ in _TTSServerStats._fields_}


def postnet_layers(sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """Picks the post-net's conv / batch-norm tensors out of a SpeechT5 state_dict, whatever prefix they carry
    (`layers.0.conv.weight`, `speech_decoder_postnet.layers.0.conv.weight`, ...)."""
    out = {}
    for k, v in sd.items():
        i = k.find("layers.")
        if i < 0 or k.endswith("num_batches_tracked"):
            continue
        if i > 0 and not k[:i].endswith("speech_decoder_postnet.") and k[:i] != "":
            continue
        tail = k[i:]
        if ".conv.weight" in tail or ".batch_norm." in tail:
            out[tail] = v
    if len(out) != 25:
        raise RuntimeError(f"post-net state_dict: expected 25 tensors (5 layers x conv.weight + 4 batch-norm tensors), found {len(out)}")
    return out


# ---- ctx-less codec / resampler calls --------------------------------------------------------------------
def _flat_rows(x: torch.Tensor):
    shape = x.shape
    return x.reshape(-1, shape[-1]) if x.dim() > 1 else x.reshape(1, -1), shape


def resample_2to1(audio: torch.Tensor) -> torch.Tensor:
    in_dtype = audio.dtype
    x = _require_cuda(audio.to(torch.float32), torch.float32, "audio")
    ensure_taps(x.device)
    rows, shape = _flat_rows(x)
    L = rows.size(1)
    out = torch.empty(rows.size(0), (L + 1) // 2, device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().b2_resample_2to1(rows.data_ptr(), rows.size(0), L, out.data_ptr(), _stream_ptr(x.device)), "resample_2to1")
    out = out.reshape(tuple(shape[:-1]) + (out.size(1),))
    return out.to(in_dtype) if in_dtype != torch.float32 else out


def resample_1to2(audio: torch.Tensor) -> torch.Tensor:
    in_dtype = audio.dtype
    x = _require_cuda(audio.to(torch.float32), torch.float32, "audio")
    ensure_taps(x.device)
    rows, shape = _flat_rows(x)
    L = rows.size(1)
    out = torch.empty(rows.size(0), 2 * L, device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().b2_resample_1to2(rows.data_ptr(), rows.size(0), L, out.data_ptr(), _stream_ptr(x.device)), "resample_1to2")
    out = out.reshape(tuple(shape[:-1]) + (2 * L,))
    return out.to(in_dtype) if in_dtype != torch.float32 else out


def g711_encode(audio: torch.Tensor, law: int = LAW_ULAW) -> torch.Tensor:
    """float (any shape, cuda) or int16 PCM -> uint8 codes, same shape."""
    lib = _lib.load()
    if not audio.is_cuda:
        raise RuntimeError("g711_encode needs a CUDA tensor (no CPU fallback)")
    out = torch.empty(audio.shape, device=audio.device, dtype=torch.uint8)
    with torch.cuda.device(audio.device):
        if audio.dtype == torch.int16:
            x = audio.contiguous()
            _lib.check(lib.b2_g711_encode_i16(x.data_ptr(), x.numel(), law, out.data_ptr(), _stream_ptr(x.device)), "g711_encode_i16")
        else:
            x = audio.to(torch.float32).contiguous()
            _lib.check(lib.b2_g711_encode_f32(x.data_ptr(), x.numel(), law, out.data_ptr(), _stream_ptr(x.device)), "g711_encode_f32")
    return out


def f32_to_pcm16(audio: torch.Tensor) -> torch.Tensor:
    x = _require_cuda(audio, torch.float32, "audio")
    out = torch.empty(x.shape, device=x.device, dtype=torch.int16)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().b2_f32_to_pcm16(x.data_ptr(), x.numel(), out.data_ptr(), _stream_ptr(x.device)), "f32_to_pcm16")
    return out


def g711_decode(codes: torch.Tensor, law: int = LAW_ULAW, dtype=torch.float32) -> torch.Tensor:
    x = _require_cuda(codes, torch.uint8, "codes")
    out = torch.empty(x.shape, device=x.device, dtype=dtype)
    with torch.cuda.device(x.device):
        if dtype == torch.int16:
            _lib.check(_lib.load().b2_g711_decode_i16(x.data_ptr(), x.numel(), law, out.data_ptr(), _stream_ptr(x.device)), "g711_decode_i16")
        elif dtype == torch.float32:
            _lib.check(_lib.load().b2_g711_decode_f32(x.data_ptr(), x.numel(), law, out.data_ptr(), _stream_ptr(x.device)), "g711_decode_f32")
        else:
            raise RuntimeError("g711_decode: dtype must be float32 or int16")
    return out


def resample_g711_encode(audio16k: torch.Tensor, law: int = LAW_ULAW) -> torch.Tensor:
    """(rows, L) fp32 @16 kHz -> (rows, ceil(L/2)) G.711 bytes @8 kHz, one fused kernel."""
    x = _require_cuda(audio16k, torch.float32, "audio16k")
    ensure_taps(x.device)
    rows, shape = _flat_rows(x)
    L = rows.size(1)
    out = torch.empty(rows.size(0), (L + 1) // 2, device=x.device, dtype=torch.uint8)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().b2_resample_g711_encode(rows.data_ptr(), rows.size(0), L, law, out.data_ptr(), _stream_ptr(x.device)), "resample_g711_encode")
    return out.reshape(tuple(shape[:-1]) + (out.size(1),))


def g711_decode_upsample(codes: torch.Tensor, law: int = LAW_ULAW) -> torch.Tensor:
    """(rows, L) G.711 bytes @8 kHz -> (rows, 2L) fp32 @16 kHz."""
    x = _require_cuda(codes, torch.uint8, "codes")
    ensure_taps(x.device)
    rows, shape = _flat_rows(x)
    L = rows.size(1)
    out = torch.empty(rows.size(0), 2 * L, device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().b2_g711_decode_upsample(rows.data_ptr(), rows.size(0), L, law, out.data_ptr(), _stream_ptr(x.device)), "g711_decode_upsample")
    return out.reshape(tuple(shape[:-1]) + (2 * L,))


def g711_decode_many(packets: Sequence[bytes], law: int = LAW_ULAW, upsample: bool = False, device=None) -> list:
    """Batched inbound decode (SURVEY section 8 f4): the RTP payloads of any number of calls -> one pinned staging buffer, one H2D,
    one kernel launch, one D2H.  Returns a list of 1-D fp32 CPU tensors (views of one pinned buffer), 8 kHz or, with upsample, 16 kHz,
    each packet zero-padded on its own like the reference's per-call G711Codec.decode (Core/Codecs/G711.py:34-47)."""
    lib = _lib.load()
    if not torch.cuda.is_available():
        raise RuntimeError("g711_decode_many needs a CUDA device (no CPU fallback)")
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    n = len(packets)
    if n == 0:
        return []
    lens = torch.tensor([len(p) for p in packets], dtype=torch.int64)
    offs = torch.zeros(n + 1, dtype=torch.int64)
    torch.cumsum(lens, 0, out=offs[1:])
    total = int(offs[-1])
    mul = 2 if upsample else 1
    out = torch.empty(total * mul, dtype=torch.float32).pin_memory()
    if total:
        src = torch.frombuffer(bytearray(b"".join(packets)), dtype=torch.uint8).pin_memory()
        ensure_taps(dev)
        with torch.cuda.device(dev):
            _lib.check(lib.b2_g711_decode_many_host(src.data_ptr(), offs.data_ptr(), n, law, 1 if upsample else 0, out.data_ptr(), _stream_ptr(dev)),
                       "g711_decode_many_host")
    o = (offs * mul).tolist()
    return [out[o[i]:o[i + 1]] for i in range(n)]


def kernel_launch_count() -> int:
    return int(_lib.load().b2_kernel_launch_count())
