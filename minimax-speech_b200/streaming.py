"""Streaming synthesis session (SURVEY.md section 8 row f-2): the hop scheduling of ``CosyVoice2Model.tts`` (stream branch,
speech/cosyvoice/cli/model.py:336-366) and ``token2wav`` (:285-319) around the drop-in ``CausalMaskedDiffWithXvec.inference``
(``streaming=True``: block-causal attention in the token encoder and in the estimator; non-final calls carry
``pre_lookahead_len`` tokens of look-ahead context), with the DAC-VAE decoder where the reference CLI still calls HiFT
(the CLI is stale with respect to the DAC-VAE latents, SURVEY section 0, so the vocoder side is ours):

* tokens arrive incrementally (``push``); a hop is synthesised as soon as ``token_hop_len + pre_lookahead_len`` new tokens
  are there (the first hop is lengthened by ``prompt_token_pad`` so that hop boundaries fall on the 25-token attention
  chunks, model.py:339-341); every call re-runs the flow on ALL tokens so far and keeps the frames past ``token_offset``
  (model.py:296, 343-352) -- the block-causal masks make the earlier frames independent of the later tokens;
* ``finish`` runs the last call with ``finalize=True`` on whatever remains (model.py:357-366);
* the DAC-VAE decoder is not causal: a chunk is decoded with ``dac_context`` latent frames of left context and the last
  ``dac_context`` frames are held back until the next call has produced their right context (HiFT's mel / source cache and
  cross-fade, model.py:298-311, play this role in the reference).  With ``dac_context`` >= the decoder's reach (15 latent
  frames, SURVEY Appendix B) the concatenated chunks equal one decode of the whole latent sequence.
"""
import math

import torch


class StreamingSession:
    token_hop_len = 25  # must match the training static_chunk_size (model.py:255-256)

    def __init__(self, flow, dac, prompt_token, prompt_feat, embedding=None, reference_mels=None, dac_context=16):
        """flow: ``front.CausalMaskedDiffWithXvec``; dac: ``dac.DACVAEDecoder``; prompt_token [1,Tp] int, prompt_feat [1,Fp,80]
        (device tensors); embedding [1,192] or reference_mels for the speaker encoder."""
        if prompt_token.dim() != 2 or prompt_token.shape[0] != 1:
            raise ValueError("prompt_token must be [1, Tp]")
        self.flow, self.dac = flow, dac
        self.prompt_token, self.prompt_feat = prompt_token, prompt_feat
        self.embedding, self.reference_mels = embedding, reference_mels
        self.device = prompt_token.device
        self.lookahead = flow.pre_lookahead_len
        self.ratio = flow.token_latent_ratio
        hop, tp = self.token_hop_len, prompt_token.shape[1]
        self.prompt_token_pad = int(math.ceil(tp / hop) * hop - tp)  # model.py:339
        self.dac_context = int(dac_context)
        self.tokens = []
        self.token_offset = 0
        self.latents = torch.zeros(1, flow.output_size, 0, device=self.device)  # every frame synthesised so far
        self.emitted = 0  # latent frames whose audio has been handed out
        self.finished = False

    # -- token2wav (model.py:285-319), flow half -------------------------------------------------------------------------
    def _flow(self, n_tokens, finalize):
        tok = torch.tensor(self.tokens[:n_tokens], dtype=torch.int64, device=self.device).unsqueeze(0)
        n = lambda t: torch.tensor([t.shape[1]], dtype=torch.int32)  # noqa: E731
        lat, _ = self.flow.inference(token=tok, token_len=n(tok), prompt_token=self.prompt_token, prompt_token_len=n(self.prompt_token),
                                     prompt_feat=self.prompt_feat, prompt_feat_len=n(self.prompt_feat), embedding=self.embedding,
                                     reference_mels=self.reference_mels, streaming=True, finalize=finalize)
        self._append(lat)

    def _append(self, lat):
        new = lat[:, :, self.token_offset * self.ratio:]  # model.py:296
        self.latents = torch.cat([self.latents, new], dim=2)

    # -- vocoder half: DAC-VAE decode with left context and a held-back tail ---------------------------------------------
    def _window(self, hold):
        """(first latent frame the decode reads, end of the frames it hands out), or None when nothing is due."""
        end = self.latents.shape[2] - hold
        if end <= self.emitted:
            return None
        return max(0, self.emitted - self.dac_context), end

    def _take(self, wav, w0, end):
        """The new samples of ``wav`` [1, n], the decode of the latent frames from ``w0`` on."""
        hop = self.dac.hop_length
        out = wav[:, (self.emitted - w0) * hop:(end - w0) * hop]
        self.emitted = end
        return out

    def _decode(self, hold):
        win = self._window(hold)
        if win is None:
            return torch.zeros(1, 0, device=self.device)
        w0, end = win
        wav = self.dac.decode(self.latents[:, :, w0:].contiguous())
        return self._take(wav[:, 0], w0, end)

    def _hop_len(self):
        return self.token_hop_len + self.prompt_token_pad if self.token_offset == 0 else self.token_hop_len

    def _next_hop(self):
        """Tokens of the next non-final hop, or None while fewer than a hop plus the look-ahead are there (model.py:343)."""
        hop = self._hop_len()
        return hop if len(self.tokens) - self.token_offset >= hop + self.lookahead else None

    def push(self, tokens):
        """Append newly generated speech tokens; returns the list of waveform chunks [1, n] that became ready."""
        if self.finished:
            raise RuntimeError("session already finished")
        self.tokens.extend(int(t) for t in tokens)
        chunks = []
        while (this_hop := self._next_hop()) is not None:
            self._flow(self.token_offset + this_hop + self.lookahead, finalize=False)
            self.token_offset += this_hop
            w = self._decode(hold=self.dac_context)
            if w.shape[1]:
                chunks.append(w)
        return chunks

    def finish(self):
        """The remaining tokens with ``finalize=True`` (model.py:357-366); returns the last waveform chunk."""
        if self.finished:
            raise RuntimeError("session already finished")
        self.finished = True
        if len(self.tokens) > self.token_offset:
            self._flow(len(self.tokens), finalize=True)
            self.token_offset = len(self.tokens)
        return self._decode(hold=0)


class StreamingBatch:
    """Many streaming sessions advanced together: each round of ``step`` runs ONE ``flow.inference_batch`` call (every
    session with a hop ready, finishing ones included) and ONE length-masked ``dac.decode`` over the sessions' decode
    windows, where N ``StreamingSession``s would make N of each.  Per session, the hops, the held-back tail and the
    chunk boundaries are those of a lone ``StreamingSession`` (whose bookkeeping each session here is), and so are the
    chunks, up to the batched flow solve's last-bit differences.  The caller serialises ``open``, ``push``, ``finish``
    and ``step``."""

    def __init__(self, flow, dac, dac_context=16):
        """flow: ``front.CausalMaskedDiffWithXvec``; dac: ``dac.DACVAEDecoder``."""
        self.flow, self.dac, self.dac_context = flow, dac, int(dac_context)
        self._sessions, self._embedding, self._finishing = {}, {}, set()
        self._next_id = 0

    def open(self, prompt_token, prompt_feat, embedding=None, reference_mels=None):
        """Starts a session (prompt_token [1,Tp] int, prompt_feat [1,Fp,80], embedding [1,192] or reference_mels for the
        speaker encoder, as ``StreamingSession``); returns its id.  The speaker embedding is computed here, once."""
        sess = StreamingSession(self.flow, self.dac, prompt_token, prompt_feat, dac_context=self.dac_context)
        sid = self._next_id
        self._next_id += 1
        self._embedding[sid] = self.flow.get_speaker_embedding(
            {"reference_mels": reference_mels, "embedding": embedding, "speech_token": prompt_token}, sess.device)
        self._sessions[sid] = sess
        return sid

    def _get(self, sid):
        if sid in self._finishing or (sid not in self._sessions and isinstance(sid, int) and 0 <= sid < self._next_id):
            raise RuntimeError(f"session {sid} already finished")
        if sid not in self._sessions:
            raise KeyError(f"no session {sid!r}")
        return self._sessions[sid]

    def push(self, sid, tokens):
        """Appends newly generated speech tokens to session ``sid``; nothing is synthesised before ``step``."""
        self._get(sid).tokens.extend(int(t) for t in tokens)

    def finish(self, sid):
        """Marks session ``sid`` complete: the next ``step`` runs its remaining hops, then its ``finalize=True`` call."""
        self._get(sid)
        self._finishing.add(sid)

    def __len__(self):
        return len(self._sessions)

    def step(self):
        """Advances every session as far as its tokens allow -> {id: [waveform chunks [1, n]]}.  A finished session's
        last chunk (possibly empty) is always there, and the session is closed with it."""
        out = {}
        while True:
            calls = {}  # sid -> (tokens the flow call covers, finalize)
            for sid, sess in self._sessions.items():
                hop = sess._next_hop()
                if hop is not None:
                    calls[sid] = (hop, False)
                elif sid in self._finishing:
                    calls[sid] = (len(sess.tokens) - sess.token_offset, True)
            if not calls:
                return out
            self._round(calls, out)

    def _round(self, calls, out):
        ss = {sid: self._sessions[sid] for sid in calls}
        flow_ids = [sid for sid, (hop, fin) in calls.items() if hop > 0]
        if flow_ids:
            dev = ss[flow_ids[0]].device
            toks, fins = [], []
            for sid in flow_ids:
                s, (hop, fin) = ss[sid], calls[sid]
                n = s.token_offset + hop + (0 if fin else s.lookahead)
                toks.append(torch.tensor(s.tokens[:n], dtype=torch.int64).to(dev))
                fins.append(fin)
            lat, lens = self.flow.inference_batch(toks, [ss[i].prompt_token for i in flow_ids], [ss[i].prompt_feat for i in flow_ids],
                                                  torch.cat([self._embedding[i] for i in flow_ids], dim=0), fins, streaming=True)
            for b, sid in enumerate(flow_ids):
                ss[sid]._append(lat[b:b + 1, :, :int(lens[b])])
                ss[sid].token_offset += calls[sid][0]
        wins = {}
        for sid, (hop, fin) in calls.items():
            w = ss[sid]._window(0 if fin else ss[sid].dac_context)
            if w is not None:
                wins[sid] = w
        if wins:
            n = [ss[sid].latents.shape[2] - w0 for sid, (w0, _) in wins.items()]
            first = ss[next(iter(wins))].latents
            z = torch.zeros(len(n), first.shape[1], max(n), device=first.device)
            for b, (sid, (w0, _)) in enumerate(wins.items()):
                z[b, :, :n[b]] = ss[sid].latents[0, :, w0:]
            wav = self.dac.decode(z, torch.tensor(n, dtype=torch.int32))
            for b, (sid, (w0, end)) in enumerate(wins.items()):
                out.setdefault(sid, []).append(ss[sid]._take(wav[b:b + 1, 0], w0, end))
        for sid, (hop, fin) in calls.items():
            if fin:
                if sid not in wins:
                    out.setdefault(sid, []).append(torch.zeros(1, 0, device=ss[sid].device))
                ss[sid].finished = True
                del self._sessions[sid], self._embedding[sid]
                self._finishing.discard(sid)
