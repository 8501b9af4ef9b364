"""The reference's nn.Module surface (model.py) over the B200 engine.

Same class names, constructor signatures, attribute names, parameter registration order (hence the
same ``state_dict`` keys AND the same random initialisation under a given torch seed) as
NVIDIA/tacotron2 ``model.py`` -- so ``train.py`` / ``inference.ipynb`` / published checkpoints work
unchanged -- but ``forward`` / ``inference`` run hand-written sm_100a kernels through libt2b200.so:

    Tacotron2.inference  (model.py:517-529)  -> encoder kernels -> persistent decoder kernel -> postnet
    Tacotron2.forward    (model.py:499-515)  -> encoder -> teacher-forced decoder -> postnet -> parse_output
    Decoder.inference    (model.py:418-454)  -> t2_decoder_run(INFER): batched, per-row stop latch
    Decoder.forward      (model.py:381-416)  -> t2_prenet_forward + t2_decoder_run(TEACHER)
    Encoder.forward/.inference (:173-201), Postnet.forward (:141-146)

There is no CPU path: calling these on CPU tensors raises.
"""
import weakref
from math import sqrt

import torch
from torch import nn

from . import _capi
from ._engine import Engine, current_masks, next_seed
from .layers import ConvNorm, LinearNorm
from .utils import get_mask_from_lengths, to_gpu


class LocationLayer(nn.Module):
    """model.py:10-26 (parameters only; evaluated inside the decoder kernels)."""

    def __init__(self, attention_n_filters, attention_kernel_size, attention_dim):
        super(LocationLayer, self).__init__()
        padding = int((attention_kernel_size - 1) / 2)
        self.location_conv = ConvNorm(2, attention_n_filters, kernel_size=attention_kernel_size,
                                      padding=padding, bias=False, stride=1, dilation=1)
        self.location_dense = LinearNorm(attention_n_filters, attention_dim, bias=False, w_init_gain='tanh')


class Attention(nn.Module):
    """model.py:29-86 (parameters + score_mask_value, which train.py:76 overwrites from outside)."""

    def __init__(self, attention_rnn_dim, embedding_dim, attention_dim, attention_location_n_filters,
                 attention_location_kernel_size):
        super(Attention, self).__init__()
        self.query_layer = LinearNorm(attention_rnn_dim, attention_dim, bias=False, w_init_gain='tanh')
        self.memory_layer = LinearNorm(embedding_dim, attention_dim, bias=False, w_init_gain='tanh')
        self.v = LinearNorm(attention_dim, 1, bias=False)
        self.location_layer = LocationLayer(attention_location_n_filters, attention_location_kernel_size,
                                            attention_dim)
        self.score_mask_value = -float("inf")


class _EngineOwner(object):
    """Mixin: finds (or lazily creates) the Engine for this module.  Sub-modules of a Tacotron2 share
    the root's engine; a stand-alone Encoder / Decoder / Postnet builds its own (the weight-table
    entries it does not have are filled with zeros)."""

    _t2_prefix = ""

    def _t2_root(self):
        ref = self.__dict__.get("_t2_root_ref")
        root = ref() if ref is not None else None
        return root if root is not None else self

    def _t2_link(self):
        """(Re-)point the children at this module as their engine owner.  The links are weak references kept out of
        copies / pickles (__getstate__ below), so they are rebuilt lazily: a deepcopy of a Tacotron2 must resolve ITS OWN
        parameters, not the original's."""
        ref = None
        for child in self._t2_children():
            cur = child.__dict__.get("_t2_root_ref")
            if cur is None or cur() is not self:
                if ref is None:
                    ref = weakref.ref(self)
                child.__dict__["_t2_root_ref"] = ref

    def _t2_children(self):
        return ()

    def __getstate__(self):
        # copy.deepcopy / pickle / torch.save(model): the engine (a ctypes handle + device workspaces) and the weak
        # back-references are per-instance runtime state; the copy builds its own on first use
        state = dict(super().__getstate__())       # nn.Module.__getstate__ (the mixin precedes nn.Module in the MRO)
        state.pop("_t2_root_ref", None)
        state.pop("_t2_engine_obj", None)
        return state

    def invalidate_weights(self):
        """Call after writing parameters / buffers in a way torch's version counter does not see (``p.data.copy_()``,
        ``p.data.mul_()``, raw pointer writes): the packed device-side operand images are rebuilt on the next call."""
        eng = self._t2_root().__dict__.get("_t2_engine_obj")
        if eng is not None:
            eng.invalidate()

    def _t2_engine(self):
        root = self._t2_root()
        root._t2_link()
        eng = root.__dict__.get("_t2_engine_obj")
        if eng is None:
            eng = Engine(root._t2_hparams)
            root.__dict__["_t2_engine_obj"] = eng
        prefix = root._t2_prefix
        if "_t2_hparams" not in root.__dict__:
            raise RuntimeError("tacotron2_b200: %s must be used as part of a Decoder / Tacotron2" % type(self).__name__)
        named = {}
        for k, v in root.named_parameters():
            named[prefix + k] = v
        for k, v in root.named_buffers():
            named[prefix + k] = v
        # under autograd in training mode the parameters change every step (possibly through .data, which the version
        # counter does not see): always re-pack there; otherwise the (pointer, version, dtype) key decides
        # ... once per top-level call: the modules Tacotron2.forward calls in turn (embedding + encoder, decoder, postnet)
        # share the packing done at its start (root._t2_packed_in_call), they do not repeat it
        force = (root.training and torch.is_grad_enabled() and not root.__dict__.get("_t2_packed_in_call", False) and
                 any(p_.requires_grad for p_ in root.parameters()))
        eng.ensure(named, force=force)
        return eng

    def _t2_out_dtype(self):
        for p_ in self.parameters():
            return p_.dtype
        return torch.float32


def _invalidate_after_load(module, incompatible_keys):
    """load_state_dict copies into the parameters through .data-like paths: re-pack on the next call."""
    module.invalidate_weights()


def _require_no_grad(module, what):
    if torch.is_grad_enabled() and any(p_.requires_grad for p_ in module.parameters()):
        raise NotImplementedError(
            "tacotron2_b200: %s on its own has no autograd node (the prenet's backward is part of Decoder.forward's, "
            "model.py:396-399); call it through Decoder.forward / Tacotron2.forward or under torch.no_grad()" % what)


def _wants_grad(module, *tensors):
    return torch.is_grad_enabled() and (any(t is not None and t.requires_grad for t in tensors) or
                                        any(p_.requires_grad for p_ in module.parameters()))


MAX_TRAIN_ROWS = 64   # rows per GPU of one autograd call: the backward kernels and the training stash are sized for one
                      # 64-row launch (BASELINE.json configs[2] / [3] are B=64 per GPU); larger batches: split and accumulate


def _check_train_rows(B, what):
    if B > MAX_TRAIN_ROWS:
        raise RuntimeError("tacotron2_b200: %s under autograd supports at most %d rows per call (got %d): run the batch as "
                           "%d-row slices and let the gradients accumulate, or wrap inference-only calls in torch.no_grad()"
                           % (what, MAX_TRAIN_ROWS, B, MAX_TRAIN_ROWS))


MAX_TRAIN_T_ENC = 408  # longest encoder sequence the decoder backward takes: att_bwd_smem(T_enc) <= 220 KiB (decoder_backward.cu)


def _check_train_t_enc(T_enc, what):
    # raised before any kernel runs, so no parameter is left with a partially accumulated .grad and no BatchNorm running
    # statistic moves for a step that cannot complete
    if T_enc > MAX_TRAIN_T_ENC:
        raise RuntimeError("tacotron2_b200: %s under autograd: T_enc = %d too long for the attention kernel of the decoder "
                           "backward (at most %d encoder positions)" % (what, T_enc, MAX_TRAIN_T_ENC))


class _EncoderFn(torch.autograd.Function):
    """Encoder.forward (model.py:173-190) [+ the embedding lookup of model.py:503 when `text` is given] as one autograd
    node: forward = fp32 conv stack + persistent BiLSTM with a stash, backward = t2_encoder_backward."""

    @staticmethod
    def forward(ctx, owner, prefix_params, text, embedded, lengths, training, *params):
        eng = owner._t2_engine()
        keep = current_masks()["enc"]
        seed = next_seed()
        src = text if text is not None else embedded
        B, T = int(src.shape[0]), int(src.shape[1])
        stash = eng.stash_buffer("encoder", B, T)
        emb32 = None
        if embedded is not None:
            emb32 = embedded.detach().to(dtype=torch.float32).contiguous()
        memory = eng.encoder(text=text, embedded=emb32, lengths=lengths, training=training, keep=keep, stash=stash, seed=seed)
        if training and not owner._t2_root().__dict__.get("_t2_packed_in_call", False):
            eng.invalidate()              # running statistics changed under the packed copies (see Tacotron2._forward_packed)
        ctx.saved = dict(eng=eng, text=text, embedded=emb32, lengths=lengths, training=training, keep=keep, seed=seed,
                         stash=stash, names=prefix_params, params=params,
                         emb_dtype=embedded.dtype if embedded is not None else None)
        return memory

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, d_memory):
        sv = ctx.saved
        f32 = dict(device=d_memory.device, dtype=torch.float32)
        grads = {n: torch.empty(p_.shape, **f32) for n, p_ in zip(sv["names"], sv["params"])}
        d_emb = sv["eng"].encoder_backward(sv["text"], sv["embedded"], sv["lengths"], sv["training"], sv["keep"], sv["seed"],
                                           sv["stash"], d_memory, sv["embedded"] is not None, grads)
        ctx.saved = None
        if d_emb is not None:
            d_emb = d_emb.to(sv["emb_dtype"])
        return (None, None, None, d_emb, None, None) + tuple(grads[n].to(p_.dtype) for n, p_ in zip(sv["names"], sv["params"]))


class _PostnetFn(torch.autograd.Function):
    """Postnet.forward (model.py:141-146) [+ the residual of model.py:511 when add_residual] as one autograd node."""

    @staticmethod
    def forward(ctx, owner, names, mel_btc, add_residual, training, wgrad_lengths, *params):
        eng = owner._t2_engine()
        keep = current_masks()["post"]
        seed = next_seed()
        x = mel_btc.detach()
        if x.dtype != torch.float32 or x.stride(2) != 1 or x.stride(1) != x.shape[2]:
            x = x.float().contiguous()
        B, T = int(x.shape[0]), int(x.shape[1])
        stash = eng.stash_buffer("postnet", B, T)
        out = eng.postnet(x, None, add_residual, training, keep, stash=stash, seed=seed)
        if training and not owner._t2_root().__dict__.get("_t2_packed_in_call", False):
            eng.invalidate()
        ctx.saved = dict(eng=eng, B=B, T=T, add_residual=add_residual, training=training, keep=keep, seed=seed, stash=stash,
                         names=names, params=params, in_dtype=mel_btc.dtype, wgrad_lengths=wgrad_lengths)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, d_out):
        sv = ctx.saved
        f32 = dict(device=d_out.device, dtype=torch.float32)
        grads = {n: torch.empty(p_.shape, **f32) for n, p_ in zip(sv["names"], sv["params"])}
        d_mel = sv["eng"].postnet_backward(sv["B"], sv["T"], sv["training"], sv["add_residual"], sv["keep"], sv["seed"],
                                           sv["stash"], d_out, grads, sv["wgrad_lengths"])
        ctx.saved = None
        return (None, None, d_mel.to(sv["in_dtype"]), None, None, None) + tuple(grads[n].to(p_.dtype) for n, p_ in
                                                                          zip(sv["names"], sv["params"]))


class Prenet(_EngineOwner, nn.Module):
    """model.py:89-100.  Dropout(0.5) is always on, as in the reference (model.py:99)."""
    _t2_prefix = "decoder.prenet."

    def __init__(self, in_dim, sizes):
        super(Prenet, self).__init__()
        in_sizes = [in_dim] + sizes[:-1]
        self.layers = nn.ModuleList(
            [LinearNorm(in_size, out_size, bias=False) for (in_size, out_size) in zip(in_sizes, sizes)])

    def forward(self, x):
        _require_no_grad(self, "Prenet.forward")
        eng = self._t2_engine()
        shp = x.shape
        keep = current_masks()["prenet"]
        if keep is not None:   # (steps, 2, B, 256) -> (2, steps*B, 256)
            keep = keep.permute(1, 0, 2, 3).reshape(2, -1, keep.shape[-1])
        out = eng.prenet(x.reshape(-1, shp[-1]), keep)
        return out.reshape(*shp[:-1], out.shape[-1]).to(x.dtype)


class Postnet(_EngineOwner, nn.Module):
    """model.py:103-146: five conv1d(k=5) + BatchNorm1d, tanh on the first four."""
    _t2_prefix = "postnet."

    def __init__(self, hparams):
        super(Postnet, self).__init__()
        self.__dict__["_t2_hparams"] = hparams
        self.convolutions = nn.ModuleList()
        self.convolutions.append(
            nn.Sequential(
                ConvNorm(hparams.n_mel_channels, hparams.postnet_embedding_dim,
                         kernel_size=hparams.postnet_kernel_size, stride=1,
                         padding=int((hparams.postnet_kernel_size - 1) / 2), dilation=1, w_init_gain='tanh'),
                nn.BatchNorm1d(hparams.postnet_embedding_dim)))
        for i in range(1, hparams.postnet_n_convolutions - 1):
            self.convolutions.append(
                nn.Sequential(
                    ConvNorm(hparams.postnet_embedding_dim, hparams.postnet_embedding_dim,
                             kernel_size=hparams.postnet_kernel_size, stride=1,
                             padding=int((hparams.postnet_kernel_size - 1) / 2), dilation=1, w_init_gain='tanh'),
                    nn.BatchNorm1d(hparams.postnet_embedding_dim)))
        self.convolutions.append(
            nn.Sequential(
                ConvNorm(hparams.postnet_embedding_dim, hparams.n_mel_channels,
                         kernel_size=hparams.postnet_kernel_size, stride=1,
                         padding=int((hparams.postnet_kernel_size - 1) / 2), dilation=1, w_init_gain='linear'),
                nn.BatchNorm1d(hparams.n_mel_channels)))

    def _run(self, x, lengths, add_residual):
        xt = x.transpose(1, 2)                       # (B, T, 80): the decoder's native storage
        if lengths is None and _wants_grad(self, x):
            named = [("postnet." + k, p_) for k, p_ in self.named_parameters()]
            return _PostnetFn.apply(self, [n for n, _ in named], xt, add_residual, self.training, None,
                                    *[p_ for _, p_ in named]).to(x.dtype)
        eng = self._t2_engine()
        if xt.dtype != torch.float32 or xt.stride(2) != 1 or xt.stride(1) != xt.shape[2]:
            xt = xt.float().contiguous()
        return eng.postnet(xt.detach(), lengths, add_residual, self.training, current_masks()["post"]).to(x.dtype)

    def forward(self, x):
        """x (B, n_mel, T) -> postnet(x) (B, n_mel, T); the caller adds the residual (model.py:511)."""
        return self._run(x, None, False)


class Encoder(_EngineOwner, nn.Module):
    """model.py:149-201: 3 x (conv1d k5 + BatchNorm1d + ReLU [+dropout]) then a BiLSTM."""
    _t2_prefix = "encoder."

    def __init__(self, hparams):
        super(Encoder, self).__init__()
        self.__dict__["_t2_hparams"] = hparams
        convolutions = []
        for _ in range(hparams.encoder_n_convolutions):
            conv_layer = nn.Sequential(
                ConvNorm(hparams.encoder_embedding_dim, hparams.encoder_embedding_dim,
                         kernel_size=hparams.encoder_kernel_size, stride=1,
                         padding=int((hparams.encoder_kernel_size - 1) / 2), dilation=1, w_init_gain='relu'),
                nn.BatchNorm1d(hparams.encoder_embedding_dim))
            convolutions.append(conv_layer)
        self.convolutions = nn.ModuleList(convolutions)
        self.lstm = nn.LSTM(hparams.encoder_embedding_dim, int(hparams.encoder_embedding_dim / 2), 1,
                            batch_first=True, bidirectional=True)

    def _run(self, x, lengths):
        emb = x.transpose(1, 2)                      # (B, T, 512) -- contiguous when x came from the embedding
        if _wants_grad(self, x):
            _check_train_rows(x.size(0), "Encoder.forward")
            named = [("encoder." + k, p_) for k, p_ in self.named_parameters()]
            return _EncoderFn.apply(self, [n for n, _ in named], None, emb, lengths, self.training,
                                    *[p_ for _, p_ in named]).to(x.dtype)
        eng = self._t2_engine()
        out = eng.encoder(embedded=emb.detach(), lengths=lengths, training=self.training, keep=current_masks()["enc"])
        return out.to(x.dtype)

    def forward(self, x, input_lengths):
        """x (B, 512, T) embedded text, input_lengths sorted descending (pack_padded_sequence
        semantics, model.py:180-188) -> (B, T, 512)."""
        return self._run(x, input_lengths)

    def inference(self, x):
        return self._run(x, None)


class Decoder(_EngineOwner, nn.Module):
    """model.py:204-454."""
    _t2_prefix = "decoder."

    def __init__(self, hparams):
        super(Decoder, self).__init__()
        self.__dict__["_t2_hparams"] = hparams
        self.n_mel_channels = hparams.n_mel_channels
        self.n_frames_per_step = hparams.n_frames_per_step
        self.encoder_embedding_dim = hparams.encoder_embedding_dim
        self.attention_rnn_dim = hparams.attention_rnn_dim
        self.decoder_rnn_dim = hparams.decoder_rnn_dim
        self.prenet_dim = hparams.prenet_dim
        self.max_decoder_steps = hparams.max_decoder_steps
        self.gate_threshold = hparams.gate_threshold
        self.p_attention_dropout = hparams.p_attention_dropout
        self.p_decoder_dropout = hparams.p_decoder_dropout

        self.prenet = Prenet(hparams.n_mel_channels * hparams.n_frames_per_step,
                             [hparams.prenet_dim, hparams.prenet_dim])
        self.attention_rnn = nn.LSTMCell(hparams.prenet_dim + hparams.encoder_embedding_dim,
                                         hparams.attention_rnn_dim)
        self.attention_layer = Attention(hparams.attention_rnn_dim, hparams.encoder_embedding_dim,
                                         hparams.attention_dim, hparams.attention_location_n_filters,
                                         hparams.attention_location_kernel_size)
        self.decoder_rnn = nn.LSTMCell(hparams.attention_rnn_dim + hparams.encoder_embedding_dim,
                                       hparams.decoder_rnn_dim, 1)
        self.linear_projection = LinearNorm(hparams.decoder_rnn_dim + hparams.encoder_embedding_dim,
                                            hparams.n_mel_channels * hparams.n_frames_per_step)
        self.gate_layer = LinearNorm(hparams.decoder_rnn_dim + hparams.encoder_embedding_dim, 1,
                                     bias=True, w_init_gain='sigmoid')
        self.mel_lengths = None        # (B,) int32 after inference(): frames per row (stop latch)
        self._t2_link()

    def _t2_children(self):
        return (self.prenet,)

    def get_go_frame(self, memory):
        """model.py:243-256."""
        return memory.new_zeros(memory.size(0), self.n_mel_channels * self.n_frames_per_step)

    def parse_decoder_inputs(self, decoder_inputs):
        """model.py:291-309: (B, n_mel, T_out) -> (T_out, B, n_mel)."""
        decoder_inputs = decoder_inputs.transpose(1, 2)
        decoder_inputs = decoder_inputs.view(decoder_inputs.size(0),
                                             int(decoder_inputs.size(1) / self.n_frames_per_step), -1)
        return decoder_inputs.transpose(0, 1)

    def _teacher_forward(self, memory, decoder_inputs, memory_lengths, keep_stash):
        """Shared by the no-grad path and _DecoderFn.forward.  Returns (mel (B,T,80), gate, align, saved)."""
        eng = self._t2_engine()
        masks = current_masks()
        go = self.get_go_frame(memory).unsqueeze(0)
        frames = torch.cat((go.float(), self.parse_decoder_inputs(decoder_inputs).float()), dim=0)   # (T+1, B, 80)
        T_mel = frames.size(0) - 1
        pk = masks["prenet"]
        if pk is not None:
            pk = pk.permute(1, 0, 2, 3).reshape(2, -1, pk.shape[-1])
        frames2d = frames.reshape(-1, frames.size(-1))
        pre_seed, dec_seed = next_seed(), next_seed()
        px = eng.prenet(frames2d, pk, seed=pre_seed)                                                 # model.py:399
        smv = float(self.attention_layer.score_mask_value)
        mem32 = memory.detach().to(dtype=torch.float32).contiguous()
        stash = eng.decoder_stash(mem32.size(0), mem32.size(1), T_mel) if keep_stash else None
        mel, gate, align, _, _ = eng.decoder(
            mem32, _capi.MODE_TEACHER, T_mel, memory_lengths=memory_lengths, teacher_prenet=px,
            training=self.training, att_keep=masks["att"], dec_keep=masks["dec"], score_mask_value=smv,
            stash=stash, seed=dec_seed)
        saved = dict(eng=eng, memory=mem32, memory_lengths=memory_lengths, frames=frames2d, pk=pk, px=px, align=align,
                     stash=stash, pre_seed=pre_seed, dec_seed=dec_seed, training=self.training, att_keep=masks["att"],
                     dec_keep=masks["dec"], smv=smv)
        return mel, gate, align, saved

    def forward(self, memory, decoder_inputs, memory_lengths):
        """Teacher-forced pass (model.py:381-416).  Returns mel (B, n_mel, T), gate (B, T),
        alignments (B, T, T_enc).  Under autograd the backward pass is libt2b200's hand-written reverse
        recurrence (t2_decoder_backward / t2_prenet_backward)."""
        dt = memory.dtype
        params = [p_ for p_ in self.parameters()]
        if torch.is_grad_enabled() and (memory.requires_grad or any(p_.requires_grad for p_ in params)):
            _check_train_rows(memory.size(0), "Decoder.forward")
            _check_train_t_enc(memory.size(1), "Decoder.forward")
            mel, gate, align = _DecoderFn.apply(self, memory, decoder_inputs, memory_lengths, *params)
        else:
            mel, gate, align, _ = self._teacher_forward(memory, decoder_inputs, memory_lengths, False)
        return mel.transpose(1, 2).to(dt), gate.to(dt), align.to(dt)

    def inference(self, memory):
        """Free-running pass (model.py:418-454), batched: per-row stop latch, see README "batched
        inference".  Returns mel (B, n_mel, T), gate (B, T, 1), alignments (B, T, T_enc); T = steps
        until every row has fired (or max_decoder_steps); ``self.mel_lengths`` holds per-row lengths."""
        eng = self._t2_engine()
        mel, gate, align, lengths, n_steps = eng.decoder(
            memory, _capi.MODE_INFER, self.max_decoder_steps, prenet_keep=current_masks()["prenet"],
            gate_threshold=self.gate_threshold)
        n = int(n_steps.item())                      # the one host sync of the whole loop (model.py:443 syncs every step)
        self.mel_lengths = lengths
        if n == self.max_decoder_steps and bool((lengths >= n).any()):
            fired = torch.sigmoid(gate[:, n - 1]) > self.gate_threshold
            if not bool(fired.all()):
                print("Warning! Reached max decoder steps")                                         # model.py:446
        dt = memory.dtype
        return (mel[:, :n].transpose(1, 2).to(dt), gate[:, :n].unsqueeze(-1).to(dt), align[:, :n].to(dt))


class _DecoderFn(torch.autograd.Function):
    """Decoder.forward (model.py:381-416) as one autograd node: forward = the persistent teacher-forced kernel with
    its training stash, backward = t2_decoder_backward + t2_prenet_backward."""

    @staticmethod
    def forward(ctx, dec, memory, decoder_inputs, memory_lengths, *params):
        mel, gate, align, saved = dec._teacher_forward(memory, decoder_inputs, memory_lengths, True)
        ctx.dec, ctx.saved = dec, saved
        ctx.mem_dtype = memory.dtype
        ctx.set_materialize_grads(False)
        return mel, gate, align

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, d_mel, d_gate, d_align):
        sv, dec = ctx.saved, ctx.dec
        eng = sv["eng"]
        align = sv["align"]
        B, T = align.shape[0], align.shape[1]
        f32 = dict(device=align.device, dtype=torch.float32)
        if d_mel is None:
            d_mel = torch.zeros(B, T, dec.n_mel_channels, **f32)
        if d_gate is None:
            d_gate = torch.zeros(B, T, **f32)
        named = [("decoder." + k, p_) for k, p_ in dec.named_parameters()]
        grads = {n: torch.empty(p_.shape, **f32) for n, p_ in named}
        d_memory, d_px = eng.decoder_backward(
            sv["memory"], sv["memory_lengths"], sv["px"], align, sv["stash"], sv["dec_seed"], sv["training"],
            sv["att_keep"], sv["dec_keep"], sv["smv"], d_mel, d_gate, d_align, grads)
        # the prenet ran over T+1 frames (model.py:396-399); the last frame's output is unused (model.py:405)
        d_out = torch.cat((d_px.reshape(-1, d_px.shape[-1]), torch.zeros(B, d_px.shape[-1], **f32)), 0)
        eng.prenet_backward(sv["frames"], sv["pk"], sv["pre_seed"], d_out, grads)
        ctx.saved = None
        return (None, d_memory.to(ctx.mem_dtype), None, None) + tuple(grads[n].to(p_.dtype) for n, p_ in named)


class Tacotron2(_EngineOwner, nn.Module):
    """model.py:457-529."""

    def __init__(self, hparams):
        super(Tacotron2, self).__init__()
        self.__dict__["_t2_hparams"] = hparams
        self.mask_padding = hparams.mask_padding
        self.fp16_run = hparams.fp16_run
        self.n_mel_channels = hparams.n_mel_channels
        self.n_frames_per_step = hparams.n_frames_per_step
        self.embedding = nn.Embedding(hparams.n_symbols, hparams.symbols_embedding_dim)
        std = sqrt(2.0 / (hparams.n_symbols + hparams.symbols_embedding_dim))
        val = sqrt(3.0) * std  # uniform bounds for std
        self.embedding.weight.data.uniform_(-val, val)
        self.encoder = Encoder(hparams)
        self.decoder = Decoder(hparams)
        self.postnet = Postnet(hparams)
        self.mel_lengths = None
        self.register_load_state_dict_post_hook(_invalidate_after_load)
        self._t2_link()

    def _t2_children(self):
        return (self.encoder, self.decoder, self.postnet, self.decoder.prenet)

    def parse_batch(self, batch):
        """model.py:473-485."""
        text_padded, input_lengths, mel_padded, gate_padded, output_lengths = batch
        # the reference reads max_len back from the GPU copy (a device sync, model.py:478); the collate function hands over
        # host tensors, so take it there and let the (pinned, non_blocking) copies overlap
        max_len = torch.max(input_lengths.data).item()
        text_padded = to_gpu(text_padded).long()
        input_lengths = to_gpu(input_lengths).long()
        mel_padded = to_gpu(mel_padded).float()
        gate_padded = to_gpu(gate_padded).float()
        output_lengths = to_gpu(output_lengths).long()
        return ((text_padded, input_lengths, mel_padded, max_len, output_lengths), (mel_padded, gate_padded))

    def parse_output(self, outputs, output_lengths=None):
        """model.py:487-497: zero mel / mel_postnet and set gate to 1e3 beyond each row's length."""
        if self.mask_padding and output_lengths is not None:
            mask = ~get_mask_from_lengths(output_lengths, outputs[0].size(2))
            mask = mask.expand(self.n_mel_channels, mask.size(0), mask.size(1))
            mask = mask.permute(1, 0, 2)
            outputs[0].data.masked_fill_(mask, 0.0)
            outputs[1].data.masked_fill_(mask, 0.0)
            outputs[2].data.masked_fill_(mask[:, 0, :], 1e3)  # gate energies
        return outputs

    def forward(self, inputs):
        """model.py:499-515."""
        text_inputs, text_lengths, mels, max_len, output_lengths = inputs
        text_lengths, output_lengths = text_lengths.data, output_lengths.data
        eng = self._t2_engine()                       # (re-)packs the weights once for the whole forward pass
        self.__dict__["_t2_packed_in_call"] = True
        try:
            return self._forward_packed(eng, text_inputs, text_lengths, mels, output_lengths)
        finally:
            self.__dict__["_t2_packed_in_call"] = False

    def _forward_packed(self, eng, text_inputs, text_lengths, mels, output_lengths):
        masks = current_masks()
        grad = _wants_grad(self)
        if grad:
            _check_train_rows(text_inputs.size(0), "Tacotron2.forward")
            _check_train_t_enc(text_inputs.size(1), "Tacotron2.forward")
        if grad:   # embedding lookup + encoder as one node (the embedding gradient comes out of t2_encoder_backward)
            named = [("embedding.weight", self.embedding.weight)] + [("encoder." + k, p_) for k, p_ in self.encoder.named_parameters()]
            memory = _EncoderFn.apply(self, [n for n, _ in named], text_inputs, None, text_lengths, self.training,
                                      *[p_ for _, p_ in named])
        else:
            memory = eng.encoder(text=text_inputs, lengths=text_lengths, training=self.training, keep=masks["enc"])
        memory = memory.to(self._t2_out_dtype())
        mel_outputs, gate_outputs, alignments = self.decoder(memory, mels, memory_lengths=text_lengths)
        mel_btc = mel_outputs.transpose(1, 2)
        if grad:
            named = [("postnet." + k, p_) for k, p_ in self.postnet.named_parameters()]
            # parse_output below zeroes the padded frames of mel_outputs in place (model.py:492); in the reference that
            # tensor is what the first postnet conv saved for its weight gradient -> reproduce (wgrad_lengths)
            wl = output_lengths if self.mask_padding else None
            mel_outputs_postnet = _PostnetFn.apply(self, [n for n, _ in named], mel_btc, True, self.training, wl,
                                                   *[p_ for _, p_ in named]).to(mel_outputs.dtype)
        else:
            if mel_btc.dtype != torch.float32 or not mel_btc.is_contiguous():
                mel_btc = mel_btc.float().contiguous()
            mel_outputs_postnet = eng.postnet(mel_btc, None, True, self.training, masks["post"]).to(mel_outputs.dtype)
        if self.training:
            for mod in self.modules():
                if isinstance(mod, nn.BatchNorm1d) and mod.num_batches_tracked is not None:
                    mod.num_batches_tracked += 1
            # the kernels updated the BatchNorm running statistics through raw pointers (no torch version bump); the
            # BN-folded inference images must not outlive them: next call re-packs
            eng.invalidate()
        outputs = [mel_outputs, mel_outputs_postnet, gate_outputs, alignments]
        cast = self.__dict__.get("_t2_cast_outputs")     # amp.initialize(opt_level="O2"): outputs in fp32 for the loss
        if cast is not None:
            outputs = [o.to(cast) for o in outputs]
        return self.parse_output(outputs, output_lengths)

    def inference(self, inputs):
        """model.py:517-529, batched.  For B > 1 frames at t >= mel_lengths[b] of mel_outputs and
        mel_outputs_postnet are zero (same convention as parse_output); ``self.mel_lengths`` holds
        the per-row lengths.  B == 1 is exactly the reference."""
        eng = self._t2_engine()
        memory = eng.encoder(text=inputs, lengths=None, training=self.training, keep=current_masks()["enc"])
        memory = memory.to(self._t2_out_dtype())     # a .half() model hands half tensors between its modules (ipynb:89-90)
        mel_outputs, gate_outputs, alignments = self.decoder.inference(memory)
        lengths = self.decoder.mel_lengths
        self.mel_lengths = lengths
        mel_btc = mel_outputs.transpose(1, 2)
        if mel_btc.dtype != torch.float32:
            mel_btc = mel_btc.float().contiguous()
        multi = inputs.size(0) > 1
        mel_outputs_postnet = eng.postnet(mel_btc, lengths if multi else None, True, self.training,
                                          current_masks()["post"]).to(mel_outputs.dtype)
        if multi:
            pad = ~get_mask_from_lengths(lengths.long(), mel_outputs.size(2))
            mel_outputs = mel_outputs.masked_fill(pad.unsqueeze(1), 0.0)
        return self.parse_output([mel_outputs, mel_outputs_postnet, gate_outputs, alignments])
