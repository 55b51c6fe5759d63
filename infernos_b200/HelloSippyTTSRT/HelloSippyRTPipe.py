"""Drop-in for the reference's batched streaming TTS engine, with the tail computed by the B200 library.

Same public names and call signatures as /root/reference/HelloSippyTTSRT/HelloSippyRTPipe.py:
  HelloSippyPlayRequest (:47-53), HelloSippyPipeState (:59-79), HelloSippyPipeStateBatched (:81-118),
  HelloSippyRTPipe(device, model, get_processor, output_sr, **kwa) (:139-189), .infer(state) (:191-240),
  .unbatch_and_dispatch(state) -> bool (:242-259), .get_voice / get_rand_voice / get_rand_voice_id (:261-272),
  class attributes chunk_size=8, pre_nframes=2, post_nframes=2, model_sr=16000 (:144-153).

What differs, by design:
  * lines 231-240 (window builder -> vocoder -> chunker -> re-assembly -> resampler) are ONE C-ABI call
    (b2_tts_tail) when output_sr == 8000; state.pre_frames lives in a per-session slot in HBM.  The three
    callables the reference holds (self.vocoder, self.chunker, self.resampler) are still there and are used,
    in the reference's own order, when output_sr == 16000 or fused=False.
  * the G.711 payload of every call is produced on the GPU in the same pass (state.g711); the reference encodes
    later, per call, on the CPU of another process (RTP/RTPOutputWorker.py:118).
  * unbatch_and_dispatch does one device->host copy per call instead of two .item() syncs and one .cpu() per session.
  * continuous batching (SURVEY section 8 f2; the reference's `mergein` is disabled, HelloSippyRTPipeTest.py:145): infer_many()
    takes any number of independently started batch states ("cohorts", each with its own front-half state and step counter)
    and runs ONE tail call over the union of their live sessions, so requests admitted while others are mid-sentence share
    the GPU pass.  InfernTTSWorker(continuous=True) drives it.
  * the decoder post-net (:230, SURVEY section 8 f3) runs on the GPU inside the same tail call when its weights are given
    (`postnet_state_dict`, or automatically when the engine loads a SpeechT5 model itself); `frontend.postnet` is then not called.
  * the autoregressive front half is reached through a small `frontend` object.  B200Frontend (SURVEY section 8 f3) runs the decoder loop of
    :195-229 -- prenet, six decoder layers with a slot KV cache, feat_out / prob_out, 16 steps per engine call -- inside the CUDA library
    (engine.TTSDecoder, b2_dec_*) and hands the frames to the tail without leaving the device.  The text encoder (:111-116, once per
    sentence) is a callable: engine.TTSEncoder (b2_enc_*, ragged: padded positions are never computed) with B200Frontend.from_state_dict or
    from_model(gpu_encoder=True), the transformers model's own encoder otherwise; the tokenizer is a host callable.  SpeechT5Frontend issues the reference's own torch calls on a transformers model; ScriptedFrontend
    replays a fixed mel plan (tests, benchmarks of the tail alone).
  * requests may ask for pre-encoded dispatch (`pre_encoded=True`): `dispatch` then receives G711AudioChunk objects (samples + the G.711 bytes
    made on the GPU in the same pass), which the payload-aware OutputMuxer carries to the RTP packetiser un-re-encoded (f1).
"""
from __future__ import annotations

import threading
import uuid
import weakref
from typing import Callable, List, Optional

import torch

from infernos_b200._lib import LAW_ALAW, LAW_ULAW
from infernos_b200.Core.AudioChunk import G711AudioChunk
from infernos_b200.engine import TTSTail


class SessCmd:
    pass


class SessSyncCmd(SessCmd):
    live: tuple

    def __init__(self, sessions):
        self.live = tuple(sorted(sessions.keys()))


class SessDispatchCmd(SessCmd):
    session: uuid.UUID

    def __init__(self, session_id: uuid.UUID):
        self.session = session_id


class HelloSippyPlayRequest(SessDispatchCmd):
    text: str
    speaker: torch.Tensor
    dispatch: Callable

    def __init__(self, session_id: uuid.UUID, text: str, speaker: torch.Tensor, dispatch: Callable,
                 dispatch_g711: Optional[Callable] = None, pre_encoded: bool = False):
        """Extensions (SURVEY section 8 f1), both optional:
        dispatch_g711: called with the G.711 payload `bytes` of exactly the samples just handed to `dispatch`, encoded on the GPU
        in the same pass.
        pre_encoded=True: `dispatch` receives a G711AudioChunk (the same 1-D CPU tensor as `.audio` + those bytes as `.payload`)
        instead of the bare tensor, which TTSSndDispatch / the payload-aware OutputMuxer / G711Codec.encode carry to the RTP
        packetiser without a second encode (RTP/RTPOutputWorker.py:118).  End of sentence is `dispatch(None)` either way."""
        self.text, self.speaker, self.dispatch, self.dispatch_g711 = text, speaker, dispatch, dispatch_g711
        self.pre_encoded = pre_encoded
        super().__init__(session_id)


def make_tensor(x):
    return torch.tensor([x], dtype=torch.long)


class HelloSippyPipeState:
    """Per-request state before batching (reference :59-79)."""

    def __init__(self, pp: "HelloSippyRTPipe", req: HelloSippyPlayRequest):
        self.session, self.dispatch = req.session, req.dispatch
        self.dispatch_g711 = getattr(req, "dispatch_g711", None)
        self.pre_encoded = bool(getattr(req, "pre_encoded", False))
        text = req.text if pp.cleanup_text is None else pp.cleanup_text(req.text)
        self.text = text
        self.inputs = pp.frontend.tokenize(text)
        self.speaker_embeddings = req.speaker
        self.encoder_attention_mask = torch.ones_like(self.inputs, dtype=torch.int)
        self.starts_at = make_tensor(pp.post_nframes // pp.reduction_factor)
        self.ends_at = make_tensor(-1)


class HelloSippyPipeStateBatched:
    """Batch state (reference :81-118).  pre_frames is a set of slots in the engine's HBM pool."""
    idx: int = 0

    def __init__(self, states: List[HelloSippyPipeState], pp: "HelloSippyRTPipe"):
        self.merge(states, pp)

    def merge(self, states: List[HelloSippyPipeState], pp: "HelloSippyRTPipe"):
        self.dispatch = [s.dispatch for s in states]
        self.dispatch_g711 = [getattr(s, "dispatch_g711", None) for s in states]
        self.pre_encoded = [bool(getattr(s, "pre_encoded", False)) for s in states]
        self.sessions = [s.session for s in states]
        self.starts_at = torch.cat([s.starts_at for s in states])      # host tensors: no per-session sync later
        self.ends_at = torch.cat([s.ends_at for s in states])
        self.slots_host = pp._alloc_slots(len(states))
        self.slots = torch.tensor(self.slots_host, dtype=torch.int32, device=pp.device)
        self._release = weakref.finalize(self, pp._free_slots, list(self.slots_host))     # also callable: state.release()
        self.audio = None
        self.g711 = None
        self.idx = 0
        pp.frontend.start(self, states)
        self.minlen, self.maxlen = pp.frontend.length_bounds(self, pp.minlenratio, pp.maxlenratio)


def _release_state(state) -> None:
    state._release()


HelloSippyPipeStateBatched.release = _release_state      # returns the state's pre_frames slots to the pool (idempotent)


class ScriptedFrontend:
    """A front half that replays a fixed mel plan, two frames per decoder step, and scripted stop steps.  Stands in for
    SpeechT5 in tests/benchmarks (the AR decoder is out of scope).  `plan` is either one (B, N, 80) tensor for a single batch
    (rows in request order) or a dict text -> ((N, 80) tensor, stop_step) from which every started batch state picks its rows,
    which is what continuous batching needs.  The replay position lives on the batch state, so several states can be in flight."""

    reduction_factor = 2
    num_mel_bins = 80

    def __init__(self, plan, stop_step: Optional[List[int]] = None, maxlen: int = 1 << 30):
        self.plan, self.maxlen = plan, maxlen
        self.stop_step = stop_step if (stop_step or isinstance(plan, dict)) else [1 << 30] * plan.size(0)

    def tokenize(self, text):
        return torch.zeros(1, 1, dtype=torch.long)

    def start(self, state, states):
        state._fe_step = 0
        if isinstance(self.plan, dict):
            rows = [self.plan[s.text] for s in states]
            n = max(r[0].size(0) for r in rows)
            state._fe_plan = torch.stack([torch.nn.functional.pad(r[0], (0, 0, 0, n - r[0].size(0))) for r in rows])
            state._fe_stop = [int(r[1]) for r in rows]
        else:
            state._fe_plan, state._fe_stop = self.plan, self.stop_step

    def length_bounds(self, state, minlenratio, maxlenratio):
        return 0, self.maxlen

    def step(self, state):
        s = state._fe_step
        state._fe_step += 1
        plan = state._fe_plan
        spectrum = plan[:, 2 * s:2 * s + 2, :]
        if spectrum.size(1) < 2:                      # past the end of the script: silence-level frames
            spectrum = torch.nn.functional.pad(spectrum, (0, 0, 0, 2 - spectrum.size(1)), value=-4.0)
        prob = torch.tensor([[1.0, 1.0] if s >= st else [0.0, 0.0] for st in state._fe_stop])
        return spectrum, prob

    def postnet(self, spectrogram):
        return spectrogram


class SpeechT5Frontend:
    """The reference's front half on a transformers SpeechT5ForTextToSpeech (context glue, plain torch):
    encoder once per batch (:111-118), then per step prenet -> wrapped_decoder(KV cache) -> feat_out / prob_out
    (:195-229) and the postnet (:230)."""

    def __init__(self, model, processor):
        self.model, self.processor = model, processor
        self.reduction_factor = model.config.reduction_factor
        self.num_mel_bins = model.config.num_mel_bins

    def tokenize(self, text):
        return self.processor(text=text, return_tensors="pt")["input_ids"]

    def start(self, state, states):
        dev = self.model.device
        n = max(s.inputs.size(1) for s in states)
        pad = lambda t: torch.nn.functional.pad(t, (0, n - t.size(1)))
        state.inputs = torch.cat([pad(s.inputs) for s in states]).to(dev)
        state.encoder_attention_mask = torch.cat([pad(s.encoder_attention_mask) for s in states]).to(dev)
        # the reference casts every speaker vector with maybe_half() (:57,75); the x-vectors and the engine default are fp32
        mdt = next(self.model.parameters()).dtype
        state.speaker_embeddings = torch.cat([s.speaker_embeddings for s in states]).to(device=dev, dtype=mdt)
        enc = self.model.speecht5.encoder(input_values=state.inputs, attention_mask=state.encoder_attention_mask, return_dict=True)
        state.encoder_last_hidden_state = enc.last_hidden_state
        state.output_sequence = enc.last_hidden_state.new_zeros(state.inputs.size(0), 1, self.num_mel_bins)
        state.past_key_values = None

    def length_bounds(self, state, minlenratio, maxlenratio):
        n = state.encoder_last_hidden_state.size(1)
        return int(n * minlenratio / self.reduction_factor), int(n * maxlenratio / self.reduction_factor)

    @torch.no_grad()
    def step(self, state):
        m = self.model
        B = state.output_sequence.size(0)
        hs = m.speecht5.decoder.prenet(state.output_sequence, state.speaker_embeddings)[:, -1:]
        out = m.speecht5.decoder.wrapped_decoder(hidden_states=hs, attention_mask=None, encoder_hidden_states=state.encoder_last_hidden_state,
                                                 encoder_attention_mask=state.encoder_attention_mask, past_key_values=state.past_key_values,
                                                 use_cache=True, output_attentions=False, return_dict=True)
        last = out.last_hidden_state[:, -1, :]
        state.past_key_values = out.past_key_values
        spectrum = m.speech_decoder_postnet.feat_out(last).view(B, self.reduction_factor, self.num_mel_bins)
        state.output_sequence = torch.cat((state.output_sequence, spectrum[:, -1:, :]), dim=1)
        prob = m.speech_decoder_postnet.prob_out(last).sigmoid()
        return spectrum, prob

    @torch.no_grad()
    def postnet(self, spectrogram):
        return self.model.speech_decoder_postnet.postnet(spectrogram)


class B200Frontend:
    """The autoregressive front half on the GPU (SURVEY section 8 f3): prenet -> six-layer decoder with a slot KV cache -> feat_out /
    prob_out run inside the CUDA library (engine.TTSDecoder, b2_dec_*), 16 steps per engine call in one C-ABI call, and the frames never leave
    the device on their way into the tail.  What the reference runs once per sentence (:111-116) is reached through two callables:
        tokenizer(text) -> (1, n) LongTensor          (the SpeechT5 processor with from_model; any callable with from_state_dict)
        encoder(input_ids, attention_mask) -> (B, L, 768) tensor
    The encoder is engine.TTSEncoder -- the text encoder inside the library, only valid tokens computed -- with from_state_dict() and with
    from_model(gpu_encoder=True); from_model() without it keeps model.speecht5.encoder(...).last_hidden_state on the transformers model.
    `mask_fn(call_index) -> (16, 2, 256) 0/1 tensor` injects the prenet's dropout keep-masks (tests); by default they are drawn on the device."""

    reduction_factor = 2
    num_mel_bins = 80
    steps_per_call = 16

    def __init__(self, decoder, tokenizer: Callable, encoder: Callable, mask_fn: Optional[Callable] = None, seed: int = 0):
        self.decoder, self._tokenize, self._encode, self.mask_fn, self.seed = decoder, tokenizer, encoder, mask_fn, seed

    @classmethod
    def from_model(cls, model, processor, device, mode="bf16", max_sessions=64, max_steps=512, max_enc_len=128, gpu_encoder=False,
                   max_tokens=16384, **kw):
        """gpu_encoder=True runs the text encoder in the library too (engine.TTSEncoder on the model's weights); the default keeps the model's
        own torch encoder."""
        from infernos_b200.engine import TTSDecoder, TTSEncoder
        sd = model.state_dict()
        dec = TTSDecoder(device, sd, mode=mode, max_sessions=max_sessions, max_steps=max_steps, max_enc_len=max_enc_len)
        if gpu_encoder:
            encode = TTSEncoder(device, sd, mode=mode, max_tokens=max_tokens, max_len=max_enc_len)
        else:
            @torch.no_grad()
            def encode(ids, mask):
                dev = next(model.parameters()).device
                return model.speecht5.encoder(input_values=ids.to(dev), attention_mask=mask.to(dev), return_dict=True).last_hidden_state
        return cls(dec, lambda text: processor(text=text, return_tensors="pt")["input_ids"], encode, **kw)

    @classmethod
    def from_state_dict(cls, sd, tokenizer: Callable, device, mode="bf16", max_sessions=64, max_steps=512, max_enc_len=128, max_tokens=16384, **kw):
        """Token ids to frames without a transformers model object: engine.TTSEncoder and engine.TTSDecoder built from one SpeechT5ForTextToSpeech
        state_dict (`speecht5.encoder.*`, `speecht5.decoder.*`, `speech_decoder_postnet.{feat_out,prob_out}.*`).  max_enc_len (<= 450) bounds
        the padded token length of a cohort; max_tokens the rows of one encoder pass."""
        from infernos_b200.engine import TTSDecoder, TTSEncoder
        dec = TTSDecoder(device, sd, mode=mode, max_sessions=max_sessions, max_steps=max_steps, max_enc_len=max_enc_len)
        try:
            enc = TTSEncoder(device, sd, mode=mode, max_tokens=max_tokens, max_len=max_enc_len)
        except Exception:
            dec.close()
            raise
        return cls(dec, tokenizer, enc, **kw)

    def close(self) -> None:
        """Frees the library handles this front half owns (the decoder, and the encoder when it is an engine.TTSEncoder)."""
        self.decoder.close()
        if hasattr(self._encode, "close"):
            self._encode.close()

    def tokenize(self, text):
        return self._tokenize(text)

    def start(self, state, states):
        n = max(s.inputs.size(1) for s in states)
        pad = lambda t: torch.nn.functional.pad(t, (0, n - t.size(1)))
        state.inputs = torch.cat([pad(s.inputs) for s in states])
        state.encoder_attention_mask = torch.cat([pad(s.encoder_attention_mask) for s in states])
        enc = self._encode(state.inputs, state.encoder_attention_mask)
        dev = self.decoder.device
        spk = torch.cat([s.speaker_embeddings for s in states]).to(device=dev, dtype=torch.float32)
        state._enc_positions = int(enc.size(1))
        state._fe_call = 0
        self.decoder.start(state.slots, enc.to(device=dev, dtype=torch.float32).contiguous(),
                           state.encoder_attention_mask.sum(dim=1).to(device=dev, dtype=torch.int32), spk)

    def length_bounds(self, state, minlenratio, maxlenratio):
        n = state._enc_positions
        # a batch keeps stepping until its last sentence has ended, i.e. up to maxlen + 2 steps rounded up to a whole call of 16: the KV cache
        # (max_steps positions) has to hold that
        cap = max(1, self.decoder.max_steps - self.steps_per_call - 4)
        return int(n * minlenratio / self.reduction_factor), min(int(n * maxlenratio / self.reduction_factor), cap)

    def call(self, state):
        """One engine call = 16 decoder steps: -> (frames (B, 32, 80) fp32 on the device, BEFORE the post-net; stop probabilities (B, 16, 2) on the host)."""
        masks = self.mask_fn(state._fe_call) if self.mask_fn is not None else None
        if masks is not None:
            masks = masks.to(self.decoder.device)
        mel, prob = self.decoder.steps(state.slots, self.steps_per_call, masks=masks, seed=self.seed)
        state._fe_call += 1
        return mel, prob.cpu()

    def postnet(self, spectrogram):
        raise RuntimeError("B200Frontend leaves the post-net to the tail call (pass postnet_state_dict to the engine)")


class HelloSippyRTPipe:
    minlenratio: float = 0.0
    maxlenratio: float = 20.0
    threshold: float = 0.5
    chunk_size: int = 8
    pre_nframes: int = 2
    post_nframes: int = 2
    model_sr: int = 16000
    output_sr: int = 16000
    default_model = "microsoft/speecht5_tts"
    cleanup_text: Optional[Callable] = None
    gpu_postnet: bool = False          # True when post-net weights were given: line :230 then runs inside the tail call

    def __init__(self, device, model=default_model, get_processor: Optional[Callable] = None, output_sr: int = output_sr, **kwa):
        """kwa (beyond the reference's cleanup_text and SpeechT5Config overrides):
          frontend            object with tokenize/start/length_bounds/step/postnet (default: SpeechT5Frontend on `model`)
          vocoder_state_dict  SpeechT5HifiGan weights (default: `microsoft/speecht5_hifigan` via transformers, needs the hub)
          chunker_state_dict  AmendmentNetwork1 weights (default: synthetic when vocoder weights are synthetic)
          postnet_state_dict  SpeechT5SpeechDecoderPostnet weights (`layers.*`): the post-net (:230) then runs inside the tail call
                              on the GPU instead of through frontend.postnet (default: taken from `model` when the engine loads it)
          mode                'bf16' (tensor cores, default — the reference runs bf16, :57) or 'fp32'
          law                 'ulaw' (default) or 'alaw' for state.g711
          max_sessions        size of the pre_frames slot pool; max_windows: workspace in 12-frame windows
          fused               False forces the three-callable path of the reference
          speaker_embeddings  list of (1,512) tensors (default: one zero vector; the x-vector dataset needs the hub)
        """
        self.cuda_lock = threading.Lock()          # the reference's process-wide torcher mutex (:156), here per engine
        self.cleanup_text = kwa.pop("cleanup_text", self.cleanup_text)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("HelloSippyRTPipe (B200) needs a CUDA device; there is no CPU fallback")
        self.output_sr = output_sr
        if output_sr not in (8000, 16000):
            raise RuntimeError("output_sr must be 8000 or 16000")
        frontend = kwa.pop("frontend", None)
        voc_sd = kwa.pop("vocoder_state_dict", None)
        chk_sd = kwa.pop("chunker_state_dict", None)
        pn_sd = kwa.pop("postnet_state_dict", None)
        mode = kwa.pop("mode", "bf16")
        self.law = {"ulaw": LAW_ULAW, "alaw": LAW_ALAW}[kwa.pop("law", "ulaw")]
        max_sessions = kwa.pop("max_sessions", 64)
        max_windows = kwa.pop("max_windows", max_sessions * 4)
        self.fused = kwa.pop("fused", True) and output_sr == 8000
        self.speaker_embeddings = kwa.pop("speaker_embeddings", None) or [torch.zeros(1, 512)]
        if frontend is None:
            frontend = self._load_speecht5(model, get_processor, kwa)
            if pn_sd is None:
                pn_sd = frontend.model.speech_decoder_postnet.state_dict()
        self.frontend = frontend
        self.reduction_factor = frontend.reduction_factor
        if voc_sd is None:
            voc_sd = self._load_hub_vocoder()
        if chk_sd is None:
            raise RuntimeError("chunker_state_dict is required (sobomax/speecht5-rt.post_vocoder.v2 cannot be fetched offline)")
        self.tail = TTSTail(self.device, voc_sd, chk_sd, mode=mode, max_sessions=max_sessions, max_windows=max_windows, postnet_sd=pn_sd)
        self.gpu_postnet = pn_sd is not None
        self.device = self.tail.device
        # the reference's three plug points (:236, :237, :240)
        self.vocoder = self.tail.vocoder
        self.chunker = self.tail.chunker
        self.resampler = self.tail.resampler if self.model_sr != output_sr else None
        self._free = list(range(max_sessions - 1, -1, -1))
        self._slot_lock = threading.Lock()

    # ---- optional loaders (need network / local HF cache; not used by tests) ------------------------------
    def _load_speecht5(self, model, get_processor, kwa):
        from transformers import SpeechT5Config, SpeechT5ForTextToSpeech, SpeechT5Processor
        mc = SpeechT5Config.from_pretrained(model, **kwa)
        proc = SpeechT5Processor.from_pretrained(model, config=mc) if get_processor is None else get_processor(self.device, model, config=mc)
        m = SpeechT5ForTextToSpeech.from_pretrained(model, config=mc).to(self.device).to(torch.bfloat16).eval()
        for p in m.parameters():
            p.requires_grad = False
        return SpeechT5Frontend(m, proc)

    def _load_hub_vocoder(self):
        from transformers import SpeechT5HifiGan
        return SpeechT5HifiGan.from_pretrained("microsoft/speecht5_hifigan").state_dict()

    # ---- slots ---------------------------------------------------------------------------------------------
    def _alloc_slots(self, n: int) -> List[int]:
        with self._slot_lock:
            if n > len(self._free):
                raise RuntimeError(f"out of session slots ({n} requested, {len(self._free)} free); raise max_sessions")
            got = [self._free.pop() for _ in range(n)]
        self.tail.reset_sessions(got)          # state.pre_frames = zeros (:77)
        return got

    def _free_slots(self, slots: List[int]) -> None:
        with self._slot_lock:
            self._free.extend(slots)

    # ---- the engine ----------------------------------------------------------------------------------------
    def _front_half(self, state: HelloSippyPipeStateBatched) -> torch.Tensor:
        """Reference :195-230 for one batch state: 16 decoder steps (32 frames), stop bookkeeping, postnet.  -> mel (B, 32, 80);
        with gpu_postnet the frames are returned as feat_out produced them and the post-net is left to the tail call."""
        eframes = self.pre_nframes + self.post_nframes
        if hasattr(self.frontend, "call"):
            # GPU front half: the 16 steps are one library call; the stop rule of :225-228 is replayed step by step on the host from one
            # copy of the stop probabilities
            spectrogram, prob = self.frontend.call(state)
            for s in range(prob.size(1)):
                stop = (prob[:, s] >= self.threshold).sum(dim=1) > 0
                fire = (state.ends_at < 0) & (state.minlen <= state.idx) & (stop | (state.maxlen <= state.idx))
                state.ends_at = torch.where(fire, state.idx + eframes // self.reduction_factor, state.ends_at)
                state.idx += 1
            if not self.gpu_postnet:
                spectrogram = self.frontend.postnet(spectrogram)
            return spectrogram.to(device=self.device, dtype=torch.float32).contiguous()
        frames = []
        nframes = 0
        while nframes < self.chunk_size * 4:
            spectrum, prob = self.frontend.step(state)
            frames.append(spectrum)
            nframes += spectrum.size(1)
            stop = (prob >= self.threshold).sum(dim=1).cpu() > 0
            fire = (state.ends_at < 0) & (state.minlen <= state.idx) & (stop | (state.maxlen <= state.idx))
            state.ends_at = torch.where(fire, state.idx + eframes // self.reduction_factor, state.ends_at)
            state.idx += 1
        spectrogram = torch.cat(frames, dim=1)
        if not self.gpu_postnet:
            spectrogram = self.frontend.postnet(spectrogram)
        return spectrogram.to(device=self.device, dtype=torch.float32).contiguous()

    def infer(self, state: HelloSippyPipeStateBatched) -> None:
        with self.cuda_lock:
            mel = self._front_half(state)
            if self.fused:
                state.g711, state.audio = self.tail.tail(state.slots, mel, law=self.law, apply_postnet=self.gpu_postnet)
            else:
                self._infer_three_callables(state, self.tail.postnet(mel) if self.gpu_postnet else mel)

    def infer_many(self, states: List[HelloSippyPipeStateBatched]) -> None:
        """Continuous batching: every state advances by one call (its own front half, its own step counter), and the tail runs
        ONCE over the union of the sessions that still have a listener.  Sessions are independent in the tail (state = one
        pre_frames slot each), so a session's audio does not depend on which other sessions share the pass."""
        if not states:
            return
        if not self.fused:
            for st in states:
                self.infer(st)
            return
        with self.cuda_lock:
            mels, slots, parts = [], [], []
            for st in states:
                mel = self._front_half(st)
                live = [i for i, d in enumerate(st.dispatch) if d is not None]
                parts.append((st, live, mel.size(0), mel.size(1)))
                if live:
                    idx = torch.tensor(live, dtype=torch.long, device=self.device)
                    mels.append(mel.index_select(0, idx))
                    slots.append(st.slots.index_select(0, idx))
            if not mels:
                return
            g711, audio = self.tail.tail(torch.cat(slots), torch.cat(mels), law=self.law, apply_postnet=self.gpu_postnet)
            row = 0
            for st, live, B, nfr in parts:
                # rows of sessions that already ended stay zero: unbatch_and_dispatch never reads them
                st.audio = audio.new_zeros(B, audio.size(1))
                st.g711 = g711.new_zeros(B, g711.size(1))
                if live:
                    idx = torch.tensor(live, dtype=torch.long, device=self.device)
                    st.audio.index_copy_(0, idx, audio[row:row + len(live)])
                    st.g711.index_copy_(0, idx, g711[row:row + len(live)])
                    row += len(live)

    def _infer_three_callables(self, state, mel):
        """Lines 231-240 of the reference, through self.vocoder / self.chunker / self.resampler."""
        B = mel.size(0)
        eframes = self.pre_nframes + self.post_nframes
        pre = torch.stack([self.tail.get_pre_frames(s) for s in state.slots_host]).to(self.device)
        spectrogram = torch.cat((pre, mel), dim=1)
        new_pre = spectrogram[:, -eframes:, :]
        for s, f in zip(state.slots_host, new_pre.cpu()):
            self.tail.set_pre_frames(s, f)
        nchunks = spectrogram.size(1) // self.chunk_size
        spectrogram = torch.cat([spectrogram[:, i * self.chunk_size:(i + 1) * self.chunk_size + eframes, :] for i in range(nchunks)], dim=0).contiguous()
        audio = self.vocoder(spectrogram)
        audio = self.chunker(spectrogram, audio)
        audio = torch.cat(audio.split(B, dim=0), dim=1)
        state.audio = self.resampler(audio) if self.resampler else audio
        state.g711 = None

    def unbatch_prepare(self, state: HelloSippyPipeStateBatched):
        """The bookkeeping half of unbatch_and_dispatch (:242-259): ONE device->host copy for the whole batch, the slice arithmetic, and the
        end-of-sentence marking (`state.dispatch[i] = None`).  -> (deliver, more): `deliver()` makes the callbacks, in the reference's
        order, and may run on another thread (InfernTTSWorker(async_dispatch=True)); `more` is the method's return value."""
        sr_rr = self.model_sr // self.output_sr
        end_idx = state.idx - 1
        stepsize = 256 * 2 // sr_rr
        actions = []
        with self.cuda_lock:
            audio = state.audio.cpu()                       # one D2H for the whole batch
            pre_enc = getattr(state, "pre_encoded", None) or [False] * len(state.dispatch)
            want_bytes = state.g711 is not None and (any(cb is not None for cb in getattr(state, "dispatch_g711", [])) or any(pre_enc))
            g711 = state.g711.cpu().numpy() if want_bytes else None
            ename = "PCMA" if self.law == LAW_ALAW else "PCMU"
            asize = audio.size(1)
            starts, ends = state.starts_at.tolist(), state.ends_at.tolist()
            idx = state.idx
            for i, dispatch in enumerate(state.dispatch):
                if dispatch is None:
                    continue
                startoff = max(0, asize - (idx - starts[i]) * stepsize)
                endoff = min(asize, asize - ((idx - ends[i]) * stepsize if ends[i] >= 0 else 0))
                assert startoff <= endoff
                ended = 0 <= ends[i] <= end_idx
                if startoff != endoff or ended:
                    cb711 = state.dispatch_g711[i] if g711 is not None else None
                    actions.append((dispatch, i, startoff, endoff, ended, g711 is not None and pre_enc[i], cb711))
                if ended:
                    state.dispatch[i] = None
            alive = (state.ends_at < 0) | (state.ends_at > end_idx)
            more = bool(alive.any())
        out_sr = self.output_sr

        def deliver():
            for dispatch, i, startoff, endoff, ended, as_chunk, cb711 in actions:
                if startoff != endoff:
                    if as_chunk:
                        dispatch(G711AudioChunk(audio[i][startoff:endoff], out_sr, g711[i, startoff:endoff].tobytes(), ename))
                    else:
                        dispatch(audio[i][startoff:endoff])
                    if cb711 is not None:
                        cb711(g711[i, startoff:endoff].tobytes())
                if ended:
                    dispatch(None)
        return deliver, more

    def unbatch_and_dispatch(self, state: HelloSippyPipeStateBatched) -> bool:
        deliver, more = self.unbatch_prepare(state)
        deliver()
        return more

    def get_rand_voice_id(self) -> int:
        return torch.randint(0, len(self.speaker_embeddings), (1,)).item()

    def get_rand_voice(self):
        s_index = self.get_rand_voice_id()
        return (self.speaker_embeddings[s_index], s_index)

    def get_voice(self, s_index: int):
        return self.speaker_embeddings[s_index]
