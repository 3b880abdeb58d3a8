"""Drop-in for the reference's model container (rnnt/model.py:6-139) whose loss path is the fused CUDA one."""
from __future__ import annotations

import torch

from .joint import JointNetwork
from .predictor import ConvPredictor, ConvPredictorStepper


def _is_conv_predictor(p) -> bool:
    """ConvPredictor-shaped (rnnt/predictor.py:189-229): decided by the attributes the decode kernels read, not by class,
    so the reference's own `rnnt.predictor.ConvPredictor` (a model built with only joint._target_ swapped) qualifies."""
    try:
        return all(hasattr(p, a) for a in ("embedding", "input_layer_norm", "linear", "output_layer_norm")) \
            and hasattr(p.conv1, "conv") and hasattr(p.conv2, "conv")
    except AttributeError:
        return False


def _is_lstm_predictor(p) -> bool:
    """LSTMPredictor-shaped (rnnt/predictor.py:84-186): stateful call `p(ids, lengths, state) -> (out, lengths, state)`."""
    return hasattr(p, "lstm_layers") and hasattr(p, "embedding")


class RNNTModel(torch.nn.Module):
    def __init__(self, predictor, encoder, joint):
        super().__init__()
        self.predictor = predictor
        self.encoder = encoder
        self.joint = joint

    @property
    def device(self):
        return next(self.parameters()).device

    def forward(self, mel_features, mel_feature_lens, input_ids, input_id_lens, blank_idx: int):
        """Same contract as rnnt/model.py:17-43 (scalar mean loss); lines 32-41 collapse into joint.loss."""
        prepended = torch.cat([torch.full((input_ids.shape[0], 1), blank_idx, dtype=input_ids.dtype,
                                          device=input_ids.device), input_ids], dim=1)      # model.py:20-21
        decoder_features = self.predictor(prepended)                                         # model.py:24
        # model.py:27-28: the (N,L,C) VIEW of the encoder's (N,C,L) output goes to the kernels as is (no transposed copy)
        audio_features = self.encoder(mel_features).permute(0, 2, 1)
        audio_feature_lens = self.encoder.calc_output_lens(mel_feature_lens)                 # model.py:29
        return self.joint.loss(audio_features, decoder_features, input_ids.int(), audio_feature_lens.int(),
                               input_id_lens.int(), blank=-1, clamp=-1, reduction="mean")

    @torch.no_grad()
    def align(self, mel_features, mel_feature_lens, input_ids, input_id_lens, blank_idx: int):
        """Forced alignment of the transcripts `input_ids`: the inputs and steps of `forward` (blank prepend, predictor,
        the encoder's permuted view, calc_output_lens), then `JointNetwork.align`.  Returns an `Alignment`: per
        utterance the frame of each token on the best path, the path's log-probability and log P(transcript | audio).
        The modules run in their current mode (call eval() to align without dropout)."""
        prepended = torch.cat([torch.full((input_ids.shape[0], 1), blank_idx, dtype=input_ids.dtype,
                                          device=input_ids.device), input_ids], dim=1)
        decoder_features = self.predictor(prepended)
        audio_features = self.encoder(mel_features).permute(0, 2, 1)
        audio_feature_lens = self.encoder.calc_output_lens(mel_feature_lens)
        return self.joint.align(audio_features, decoder_features, input_ids.int(), audio_feature_lens.int(),
                                input_id_lens.int(), blank=-1)

    @torch.no_grad()
    def greedy_decode_features(self, audio_features, audio_feature_lens, max_length: int = 200,
                               max_outputs_per_step: int = 10, return_margins: bool = False,
                               use_cuda_graph: bool = True, sync_every: int = 16, engine: str = "kernel",
                               return_hypotheses: bool = False):
        """Batched greedy decode on given encoder features (B,T,H) with per-utterance lengths.

        Same per-utterance algorithm as rnnt/model.py:90-128 (blank or 10 emits advances the frame; stop at T_b or
        when len(tokens) incl. the seed blank reaches max_length), run for the whole batch at once with ALL loop state
        on the device: per step one joint+argmax kernel call for the batch, one incremental predictor update, and a
        handful of elementwise ops.  engine="kernel" (default) runs everything inside ONE persistent cooperative CUDA
        kernel (`rnnt_b200_greedy_decode`); engine="graph" replays a captured CUDA graph of torch ops + the argmax
        kernel per step and checks for completion every `sync_every` steps (kept as an independent cross-check and
        for joints with audio_ln / text_ln).  The reference syncs on `.item()` every step (model.py:113).
        return_hypotheses=True (kernel engine only) returns one `DecodedHypothesis` per utterance: tokens with their
        frames and log-probabilities, and the greedy path's score."""
        if not audio_features.is_cuda:
            raise RuntimeError("rnnt_b200 decode runs on CUDA tensors only; there is no CPU fallback")
        if _is_lstm_predictor(self.predictor):
            if return_margins:
                raise ValueError("return_margins is only available with a ConvPredictor")
            if return_hypotheses:
                raise ValueError("return_hypotheses is only available with a ConvPredictor")
            return self._greedy_decode_features_stateful(audio_features, audio_feature_lens, max_length,
                                                         max_outputs_per_step)
        if not _is_conv_predictor(self.predictor):
            raise ValueError("Unknown predictor type")                  # rnnt/model.py:139
        if engine == "kernel" and not hasattr(self.joint, "audio_ln") and not hasattr(self.joint, "text_ln"):
            # the whole loop (joint step, argmax, per-utterance state, incremental predictor) in one persistent kernel
            from .functional import greedy_decode
            return greedy_decode(audio_features, audio_feature_lens, self.joint.joint_ln.weight,
                                 self.joint.joint_ln.bias, self.predictor, self.joint.blank_idx, max_length,
                                 max_outputs_per_step, return_margins, return_hypotheses)
        if return_hypotheses:
            raise ValueError("return_hypotheses needs engine='kernel' and a joint without audio_ln / text_ln")
        was_training = self.predictor.training
        self.predictor.eval()
        try:
            key = (tuple(audio_features.shape), str(audio_features.device), int(max_length), int(max_outputs_per_step),
                   bool(return_margins), bool(use_cuda_graph))
            sessions = self.__dict__.setdefault("_decode_sessions", {})
            sess = sessions.get(key)
            if sess is None:
                if len(sessions) >= 4:
                    sessions.clear()
                sess = sessions[key] = _DecodeSession(self, audio_features, max_length, max_outputs_per_step,
                                                      return_margins, use_cuda_graph)
            return sess.run(audio_features, audio_feature_lens, sync_every)
        finally:
            self.predictor.train(was_training)

    def streaming_decoder(self, slots: int, max_length: int = 200, max_outputs_per_step: int = 10):
        """A `StreamingGreedyDecoder` over this model's joint and (ConvPredictor-shaped) predictor with `slots` streams:
        feed it the encoder's output chunk by chunk (e.g. from `AudioEncoder.streaming_forward`)."""
        from .functional import StreamingGreedyDecoder
        return StreamingGreedyDecoder(self.joint, self.predictor, slots, max_length, max_outputs_per_step)

    @torch.no_grad()
    def beam_search_features(self, audio_features, audio_feature_lens, beam_size: int = 4, max_length: int = 200,
                             return_hypotheses: bool = False):
        """Batched beam search on given encoder features (B,T,H) (e.g. the permuted view of the encoder's (B,H,T)
        output) with per-utterance lengths, in one persistent CUDA kernel (`functional.beam_decode`): per utterance,
        up to beam_size (tokens, log-score) pairs, best first; with return_hypotheses, `DecodedHypothesis` objects
        that also carry each token's frame and log-probability."""
        from .functional import _check_kernel_decode_modules, _require_cuda, beam_decode
        _check_kernel_decode_modules(self.joint, self.predictor, "beam search")
        _require_cuda(audio_features, self.joint.joint_ln.weight)
        return beam_decode(audio_features, torch.as_tensor(audio_feature_lens), self.joint.joint_ln.weight,
                           self.joint.joint_ln.bias, self.predictor, self.joint.blank_idx, beam_size, max_length,
                           return_hypotheses)

    @torch.no_grad()
    def beam_search(self, mel_features, mel_feature_lens, beam_size: int = 4, max_length: int = 200,
                    return_hypotheses: bool = False):
        """Beam search from mel features: the encoder and its output lengths first, then `beam_search_features`."""
        audio_features = self.encoder(mel_features).permute(0, 2, 1)
        audio_feature_lens = self.encoder.calc_output_lens(mel_feature_lens)
        return self.beam_search_features(audio_features, audio_feature_lens, beam_size, max_length, return_hypotheses)

    @torch.no_grad()
    def _greedy_decode_features_hostloop(self, audio_features, audio_feature_lens, max_length: int = 200,
                                         max_outputs_per_step: int = 10):
        """Host-driven variant (one device sync per step, predictor re-run on 7-token windows); kept as an independent
        cross-check of the device-side loop in the tests."""
        dev = audio_features.device
        B, T, _ = audio_features.shape
        blank = self.joint.blank_idx
        lens = [int(x) for x in audio_feature_lens.tolist()]
        tokens = [[blank] for _ in range(B)]
        t_idx = [0] * B
        per = [0] * B
        was_training = self.predictor.training
        self.predictor.eval()
        try:
            with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
                feats = self.predictor(torch.full((B, 1), blank, dtype=torch.int64, device=dev))[:, -1, :].contiguous()
                active = [b for b in range(B) if t_idx[b] < lens[b] and len(tokens[b]) < max_length]
                while active:
                    idx = torch.tensor(active, device=dev)
                    tt = torch.tensor([t_idx[b] for b in active], device=dev)
                    toks = self.joint.argmax_step(audio_features[idx, tt], feats[idx]).tolist()
                    emitted = []
                    for j, b in enumerate(active):
                        if toks[j] == blank or per[b] >= max_outputs_per_step:
                            t_idx[b] += 1
                            per[b] = 0
                        else:
                            tokens[b].append(toks[j])
                            per[b] += 1
                            emitted.append(b)
                    by_len = {}
                    for b in emitted:
                        by_len.setdefault(min(len(tokens[b]), ConvPredictor.RECEPTIVE_FIELD), []).append(b)
                    for wl, group in by_len.items():
                        win = torch.tensor([tokens[b][-wl:] for b in group], dtype=torch.int64, device=dev)
                        feats[torch.tensor(group, device=dev)] = self.predictor(win)[:, -1, :]
                    active = [b for b in active if t_idx[b] < lens[b] and len(tokens[b]) < max_length]
        finally:
            self.predictor.train(was_training)
        return [tk[1:] for tk in tokens]

    @torch.no_grad()
    def _greedy_decode_features_stateful(self, audio_features, audio_feature_lens, max_length: int = 200,
                                         max_outputs_per_step: int = 10):
        """LSTM-predictor variant (rnnt/model.py:46-87): the recurrent state lives in the predictor's own (list of
        lists of) tensors, so the loop stays on the host, one utterance at a time as in the reference; the joint step
        + argmax of every iteration is this repo's CUDA kernel (`JointNetwork.argmax_step`).  The reference marks the
        LSTM predictor as unused for training (SURVEY 2.1); it is supported for decode parity only."""
        dev = audio_features.device
        blank = self.joint.blank_idx
        lens = [int(x) for x in audio_feature_lens.tolist()]
        was_training = self.predictor.training
        self.predictor.eval()
        results = []
        try:
            for b in range(audio_features.shape[0]):
                tokens = [blank]
                t, per = 0, 0
                ids = torch.tensor([tokens], dtype=torch.int64, device=dev)
                feats, _, state = self.predictor(ids, torch.tensor([1], dtype=torch.int64, device=dev))
                while t < lens[b] and len(tokens) < max_length:
                    tok = int(self.joint.argmax_step(audio_features[b, t:t + 1], feats[:, -1, :].contiguous())[0])
                    if tok == blank or per >= max_outputs_per_step:
                        t += 1
                        per = 0
                    else:
                        tokens.append(tok)
                        ids = torch.tensor([[tok]], dtype=torch.int64, device=dev)     # model.py:78: last token + state
                        feats, _, state = self.predictor(ids, torch.tensor([len(tokens)], dtype=torch.int64, device=dev),
                                                         state)
                        per += 1
                results.append(tokens[1:])
        finally:
            self.predictor.train(was_training)
        return results

    @torch.no_grad()
    def greedy_decode(self, mel_features, mel_feature_lens, max_length: int = 200):
        """Reference signature (rnnt/model.py:130-139): batch of one, returns list[int]; dispatches on the predictor's
        shape (ConvPredictor -> persistent kernel, LSTMPredictor -> stateful host loop), ValueError otherwise."""
        assert mel_features.shape[0] == 1, "Greedy decoding only works with a batch size of 1"
        audio_features = self.encoder(mel_features).permute(0, 2, 1).contiguous()
        # the reference loops to audio_features.shape[1] (model.py:56,100), not to the computed length
        lens = torch.tensor([audio_features.shape[1]])
        return self.greedy_decode_features(audio_features, lens, max_length)[0]


class _DecodeSession:
    """Device-resident state of one batched greedy decode (shape-specific) plus the CUDA graph of one step."""

    def __init__(self, model, audio_features, max_length, max_per_step, want_margins, use_graph):
        from .functional import joint_argmax_scratch
        self.model = model
        dev = audio_features.device
        B, T, _ = audio_features.shape
        self.B, self.T, self.dev = B, T, dev
        self.max_length, self.max_per_step = max_length, max_per_step
        self.blank = model.joint.blank_idx
        V = model.joint.joint_ln.weight.shape[0]
        i64 = dict(dtype=torch.int64, device=dev)
        self.audio = torch.empty_like(audio_features, memory_format=torch.contiguous_format)
        self.lens = torch.zeros(B, **i64)
        self.rows = torch.arange(B, device=dev)
        self.t_idx = torch.zeros(B, **i64)
        self.per = torch.zeros(B, **i64)
        self.ntok = torch.ones(B, **i64)                               # counts the seed blank (model.py:53,64)
        self.out = torch.full((B, max(max_length, 1)), self.blank, **i64)
        self.stepper = ConvPredictorStepper(model.predictor, B, dev)
        self.feats = torch.zeros(B, model.joint.joint_ln.weight.shape[1], device=dev)
        self.tok32 = torch.empty(B, dtype=torch.int32, device=dev)
        self.margin = torch.empty(B, dtype=torch.float32, device=dev)
        self.scratch = joint_argmax_scratch(B, V, dev)
        self.max_steps = T + max_length + 1
        self.margin_log = torch.full((self.max_steps, B), float("inf"), device=dev) if want_margins else None
        self.step_no = torch.zeros((), **i64)
        self.inf_row = torch.full((B,), float("inf"), device=dev)
        self.all_rows = torch.ones(B, dtype=torch.bool, device=dev)
        self.seed = torch.full((B,), self.blank, **i64)
        self.use_graph = use_graph
        self.graph = None

    def _reset(self, audio_features, lens):
        self.audio.copy_(audio_features)
        self.lens.copy_(lens.to(self.dev, torch.int64).clamp(max=self.T))
        self.t_idx.zero_(); self.per.zero_(); self.ntok.fill_(1); self.out.fill_(self.blank); self.step_no.zero_()
        if self.margin_log is not None:
            self.margin_log.fill_(float("inf"))
        self.stepper.refresh()
        self.feats.copy_(self.stepper.advance(self.seed, self.all_rows))     # predictor([blank]) (model.py:97-106)

    def _one_step(self):
        m, T = self.model, self.T
        active = (self.t_idx < self.lens) & (self.ntok < self.max_length)
        a_rows = self.audio[self.rows, self.t_idx.clamp(max=T - 1)]
        m.joint.argmax_step(a_rows, self.feats, return_margin=True, out=self.tok32, margin_out=self.margin,
                            scratch=self.scratch)
        tok = self.tok32.to(torch.int64)
        advance = active & ((tok == self.blank) | (self.per >= self.max_per_step))
        emit = active & ~advance
        if self.margin_log is not None:
            self.margin_log[self.step_no.clamp(max=self.max_steps - 1)] = torch.where(active, self.margin, self.inf_row)
            self.step_no.add_(1)
        self.t_idx.add_(advance.to(torch.int64))
        self.per.copy_(torch.where(advance, torch.zeros_like(self.per), self.per + emit.to(torch.int64)))
        pos = (self.ntok.clamp(max=self.out.shape[1]) - 1).clamp(min=0)      # k-th emitted token -> column k
        self.out[self.rows, pos] = torch.where(emit, tok, self.out[self.rows, pos])
        self.ntok.add_(emit.to(torch.int64))
        self.feats.copy_(torch.where(emit.view(-1, 1), self.stepper.advance(tok, emit), self.feats))

    def _capture(self):
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            self._one_step()                                           # warm-up outside capture
        torch.cuda.current_stream(self.dev).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self._one_step()
        self.graph = graph

    def run(self, audio_features, lens, sync_every):
        with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
            if self.use_graph and self.graph is None:
                self._reset(audio_features, lens)
                try:
                    self._capture()
                except Exception:
                    self.graph, self.use_graph = None, False
            self._reset(audio_features, lens)
            limit = int(self.lens.max()) + self.max_length + 1
            done = 0
            while done < limit:
                for _ in range(min(sync_every, limit - done)):
                    if self.graph is not None:
                        self.graph.replay()
                    else:
                        self._one_step()
                    done += 1
                if not bool(((self.t_idx < self.lens) & (self.ntok < self.max_length)).any()):
                    break
        n = (self.ntok - 1).tolist()
        out_host = self.out.tolist()
        result = [out_host[b][: n[b]] for b in range(self.B)]
        if self.margin_log is not None:
            ml = self.margin_log[:done].t().tolist()
            return result, [[x for x in ml[b] if x != float("inf")] for b in range(self.B)]
        return result


def enable_zero_edit_mode(joint: JointNetwork, enabled: bool = True) -> None:
    """Make the UNMODIFIED reference rnnt/model.py:32-41 run fused: joint.forward hands a lazy handle to a patched
    torchaudio.functional.rnnt_loss.  Call once after building the model."""
    import torchaudio
    from . import functional
    joint.zero_edit_mode = enabled
    if enabled and getattr(torchaudio.functional, "_rnnt_b200_original_rnnt_loss", None) is None:
        original = torchaudio.functional.rnnt_loss

        def patched(logits, targets, logit_lengths, target_lengths, blank=-1, clamp=-1, reduction="mean",
                    fused_log_softmax=True):
            from .joint import LazyJointLogits
            if isinstance(logits, LazyJointLogits):
                return functional.rnnt_loss(logits, targets, logit_lengths, target_lengths, blank, clamp, reduction)
            return original(logits, targets, logit_lengths, target_lengths, blank, clamp, reduction,
                            fused_log_softmax)

        torchaudio.functional._rnnt_b200_original_rnnt_loss = original
        torchaudio.functional.rnnt_loss = patched
