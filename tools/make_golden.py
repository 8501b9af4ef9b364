"""Generates tests/golden/*.npz by executing the UNMODIFIED reference model.py (a checkout of NVIDIA/tacotron2 named by
T2_REFERENCE_DIR).  Run:  T2_REFERENCE_DIR=<checkout> python tools/make_golden.py [stft | full | grads | refs]

Every file holds the inputs' seeds, the reference outputs and a checksum of the synthetic weights
(tests/common.synth_state_dict) so a drift of the generator is detected instead of silently
mis-comparing.  The reference ships no golden vectors of its own (SURVEY.md section 4); these files
are outputs of the reference itself and are what pins oracle/ and the CUDA path.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.ref_import import (REFERENCE_DIR, MaskInjector, default_hparams, import_reference_model,  # noqa: E402
                               injected_dropout)
from tests.common import (GOLDEN_DIR, collate_batches, keep_mask, rand_text, stft_inputs, synth_state_dict,  # noqa: E402
                          tensor_digest, weights_checksum)

torch.set_num_threads(8)
ref = import_reference_model()


def build(sd, training=False):
    model = ref.Tacotron2(default_hparams())
    model.load_state_dict(sd)
    return model.train(training)


def ref_batched_inference(model, text, keep, thr, max_steps):
    """Reference modules driven by a loop that mirrors model.py:435-449 row-wise (the reference's
    own Decoder.inference raises for B > 1, SURVEY.md section 3.1)."""
    dec = model.decoder
    B = text.shape[0]
    masks = [keep[t, l].bool() for t in range(max_steps) for l in range(2)]
    with torch.no_grad(), injected_dropout(ref, MaskInjector(masks)):
        emb = model.embedding(text).transpose(1, 2)
        memory = model.encoder.inference(emb)
        x = dec.get_go_frame(memory)
        dec.initialize_decoder_states(memory, mask=None)
        mels, gates, aligns = [], [], []
        done = torch.zeros(B, dtype=torch.bool); lengths = torch.zeros(B, dtype=torch.int32)
        while True:
            x = dec.prenet(x)
            mel, gate, aw = dec.decode(x)
            mels.append(mel); gates.append(gate); aligns.append(aw)
            fire = (torch.sigmoid(gate.data[:, 0]) > thr) & ~done
            lengths[fire] = len(mels); done |= fire
            if bool(done.all()) or len(mels) == max_steps:
                break
            x = mel
        lengths[~done] = len(mels)
        mel, gate, align = dec.parse_decoder_outputs(mels, gates, aligns)
        mel_masked = mel.clone()
        if B > 1:
            pad = torch.arange(mel.shape[2])[None, :] >= lengths[:, None]
            mel_masked = mel.masked_fill(pad[:, None, :], 0.0)
        post = mel_masked + model.postnet(mel_masked)
        if B > 1:
            post = post.masked_fill(pad[:, None, :], 0.0)
    return memory, mel, mel_masked, post, gate, align, lengths


def calibrate_gate(sd, text, keep, steps, quantile):
    """Pick the gate weight sign and bias so rows stop at different, non-trivial steps: the sign
    makes the gate trend upwards over time, the bias puts the threshold at ``quantile`` of the
    gate values seen after the first 4 steps."""
    sd = dict(sd); sd["decoder.gate_layer.linear_layer.bias"] = torch.zeros(1)
    model = build(sd)
    _, _, _, _, gate, _, _ = ref_batched_inference(model, text, keep, 2.0, steps)
    g = gate[:, :, 0]
    sign = 1.0 if float(g[:, steps // 2:].mean()) > float(g[:, :4].mean()) else -1.0
    g = g * sign
    return sign, -float(torch.quantile(g[:, 4:].flatten(), quantile))


def save(name, **arrays):
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    out = {}
    for k, v in arrays.items():
        out[k] = v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)
    path = os.path.join(GOLDEN_DIR, name + ".npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def infer_case(name, B, T_text, max_steps, quantile, wseed, tseed, mseed, wscale=2.0):
    sd = synth_state_dict(wseed, scale=wscale)
    text = rand_text(B, T_text, tseed)
    keep = keep_mask((max_steps, 2, B, 256), 0.5, mseed)
    best = None
    for qq in (quantile, quantile - 0.03, quantile + 0.02, quantile - 0.06, quantile + 0.04):
        sign, bias = calibrate_gate(sd, text, keep, max_steps, qq)
        sd_q = synth_state_dict(wseed, gate_bias=bias, scale=wscale, gate_sign=sign)
        r = ref_batched_inference(build(sd_q), text, keep, 0.5, max_steps)
        lengths, gate = r[6], r[4]
        live = torch.arange(gate.shape[1])[None, :] < lengths[:, None]     # decisions that matter
        margin = float((torch.sigmoid(gate[:, :, 0]) - 0.5).abs()[live].min())
        varied = len(set(lengths.tolist())) > 1 or B == 1
        score = margin if (varied and int(lengths.min()) > 2) else margin * 1e-3
        if best is None or score > best[0]:
            best = (score, sign, bias, sd_q, r, margin)
    _, sign, bias, sd, (memory, mel, mel_masked, post, gate, align, lengths), margin = best
    model = build(sd)
    if B == 1:   # cross-check against the reference's OWN inference() entry point
        model.decoder.max_decoder_steps = max_steps
        masks = [keep[t, l].bool() for t in range(max_steps) for l in range(2)]
        with torch.no_grad(), injected_dropout(ref, MaskInjector(masks)):
            o = model.inference(text)
        assert torch.equal(o[0], mel) and torch.equal(o[1], post) and torch.equal(o[3], align)
        assert torch.equal(o[2], gate)
    print(name, "lengths", lengths.tolist(), "steps", mel.shape[2], "gate margin", margin)
    save(name, B=B, T_text=T_text, max_steps=max_steps, wseed=wseed, wscale=wscale, tseed=tseed, mseed=mseed,
         gate_bias=bias, gate_sign=sign, wsum=weights_checksum(sd), memory=memory, mel=mel, mel_masked=mel_masked,
         mel_post=post, gate=gate, align=align, mel_lengths=lengths, gate_margin=margin)


def ref_free_running(model, text, keep, steps):
    """The reference's own prenet / decode modules for exactly `steps` steps, no stop test (rows are independent,
    so the trajectory of a row does not depend on when other rows stop): (memory, mel (B,80,S), gate (B,S), align)."""
    dec = model.decoder
    masks = [keep[t, l].bool() for t in range(steps) for l in range(2)]
    with torch.no_grad(), injected_dropout(ref, MaskInjector(masks)):
        emb = model.embedding(text).transpose(1, 2)
        memory = model.encoder.inference(emb)
        x = dec.get_go_frame(memory)
        dec.initialize_decoder_states(memory, mask=None)
        mels, gates, aligns = [], [], []
        for _ in range(steps):
            x = dec.prenet(x)
            mel, gate, aw = dec.decode(x)
            mels.append(mel); gates.append(gate); aligns.append(aw)
            x = mel
        mel, gate, align = dec.parse_decoder_outputs(mels, gates, aligns)
    return memory, mel, gate[:, :, 0], align


def pick_gate(gate, S):
    """Gate sign and bias (applied to decoder.gate_layer; the gate is not fed back, so the mel trajectory does not depend
    on them) such that rows stop at many different steps, at least one row never fires (the run keeps all S steps) and the
    smallest |gate pre-activation| over the live decisions -- the distance of a stop decision from flipping -- is as
    large as possible.  Only the running maxima of a row matter (a row fires at the first step whose gate exceeds the
    level), so the optimum is the midpoint of the widest gap between consecutive record values that satisfies the
    constraints: exact search, no grid."""
    best = None
    B = gate.shape[0]
    for sign in (1.0, -1.0):
        g = gate.double() * sign
        cm = torch.cummax(g, dim=1)[0]
        rec = torch.unique(cm.flatten())                       # sorted record values of all rows
        gaps = rec[1:] - rec[:-1]
        for j in torch.argsort(gaps, descending=True)[:2000].tolist():
            level = 0.5 * float(rec[j] + rec[j + 1])
            fired = cm > level
            never = ~fired.any(1)
            lengths = torch.where(never, torch.full((B,), S), fired.float().argmax(1) + 1)
            n_never = int(never.sum())
            if n_never < 1 or n_never > B // 4 or int(lengths.min()) < 8 or len(set(lengths.tolist())) < B // 2:
                continue
            live = torch.arange(S)[None, :] < lengths[:, None]
            margin = float((g - level).abs()[live].min())
            if best is None or margin > best[0]:
                best = (margin, sign, -level, lengths.to(torch.int32))
            break                                              # gaps are sorted: the first feasible one is the widest
    assert best is not None, "no gate calibration found"
    return best


# frames / alignment rows kept by the full-size fixtures: sparse enough that each file stays under 1 MB
FULL_STRIDE, FULL_TAIL, FULL_ALIGN_STRIDE = 50, 8, 200


def full_frame_index(S, stride=FULL_STRIDE):
    return sorted(set(range(0, S, stride)) | set(range(S - FULL_TAIL, S)))


def full_infer_case(name, B, T_text, S, wseed, tseed, mseed, wscale):
    """The configuration a number is QUOTED on (BASELINE.json configs[1] / configs[4] per GPU), all S steps through the
    reference's own modules.  Stored: every 50th frame + the last 8 of mel / mel_postnet, all gates, all mel_lengths,
    the alignment argmax of every step and the alignment rows of every 200th step."""
    sd0 = synth_state_dict(wseed, gate_bias=0.0, scale=wscale)
    text = rand_text(B, T_text, tseed)
    keep = keep_mask((S, 2, B, 256), 0.5, mseed)
    memory, mel, gate0, align = ref_free_running(build(sd0), text, keep, S)
    margin, sign, bias, lengths = pick_gate(gate0, S)
    sd = synth_state_dict(wseed, gate_bias=bias, scale=wscale, gate_sign=sign)
    model = build(sd)
    with torch.no_grad():
        gate = model.decoder.gate_layer.linear_layer.bias + sign * gate0        # what the calibrated reference outputs
        pad = torch.arange(S)[None, :] >= lengths[:, None]
        mel_masked = mel.masked_fill(pad[:, None, :], 0.0)
        post = (mel_masked + model.postnet(mel_masked)).masked_fill(pad[:, None, :], 0.0)
    if B <= 8 or os.environ.get("T2_GOLDEN_VERIFY", "1") == "1":   # the calibrated model, stop test on, gives the same thing
        r = ref_batched_inference(model, text, keep, 0.5, S)
        assert r[6].tolist() == lengths.tolist(), (r[6].tolist(), lengths.tolist())
        assert torch.equal(r[1], mel) and torch.equal(r[3], post) and torch.allclose(r[4][:, :, 0], gate, atol=1e-6)
        gate = r[4][:, :, 0]
    idx = torch.tensor(full_frame_index(S))
    aidx = torch.arange(0, S, FULL_ALIGN_STRIDE)
    print(name, "lengths min/max", int(lengths.min()), int(lengths.max()), "distinct", len(set(lengths.tolist())),
          "gate pre-activation margin %.3e" % margin)
    save(name, B=B, T_text=T_text, max_steps=S, wseed=wseed, wscale=wscale, tseed=tseed, mseed=mseed, gate_bias=bias,
         gate_sign=sign, wsum=weights_checksum(sd), frame_index=idx, align_index=aidx, mel_masked=mel_masked[:, :, idx],
         mel_post=post[:, :, idx], gate=gate, mel_lengths=lengths, gate_margin=margin,
         align_argmax=align.argmax(-1).to(torch.int16), align_max=align.max(-1)[0], align_rows=align[:, aidx],
         memory_abs_sum=memory.double().abs().sum())


def forward_case(name, training, B, T_text, T_mel, wseed, seed, wscale=2.0):
    sd = synth_state_dict(wseed, scale=wscale)
    g = torch.Generator().manual_seed(seed)
    text = rand_text(B, T_text, seed + 1)
    tl = torch.sort(torch.randint(T_text // 3, T_text + 1, (B,), generator=g), descending=True)[0]
    tl[0] = T_text
    ol = torch.randint(T_mel // 3, T_mel + 1, (B,), generator=g); ol[1] = T_mel
    mels = torch.randn(B, 80, T_mel, generator=g)
    pk = keep_mask((T_mel + 1, 2, B, 256), 0.5, seed + 2)
    ak = keep_mask((T_mel, B, 1024), 0.1, seed + 3)
    dk = keep_mask((T_mel, B, 1024), 0.1, seed + 4)
    ek = keep_mask((3, B, 512, T_text), 0.5, seed + 5)
    qk4 = keep_mask((4, B, 512, T_mel), 0.5, seed + 6)
    qk1 = keep_mask((B, 80, T_mel), 0.5, seed + 7)
    model = build(sd, training)
    if training:
        masks = [ek[i].bool() for i in range(3)] + [pk[:, 0].bool(), pk[:, 1].bool()]
        for t in range(T_mel):
            masks += [ak[t].bool(), dk[t].bool()]
        masks += [qk4[i].bool() for i in range(4)] + [qk1.bool()]
    else:
        masks = [pk[:, 0].bool(), pk[:, 1].bool()]
    with torch.no_grad(), injected_dropout(ref, MaskInjector(masks)) as inj:
        emb = model.embedding(text).transpose(1, 2)
    with torch.no_grad(), injected_dropout(ref, MaskInjector(masks)) as inj:
        out = model((text, tl, mels, int(tl.max()), ol))
        assert inj.calls == len(masks)
    sd_after = model.state_dict()
    save(name, training=int(training), B=B, T_text=T_text, T_mel=T_mel, wseed=wseed, seed=seed, wscale=wscale,
         wsum=weights_checksum(sd), text_lengths=tl, output_lengths=ol, mels_in=mels,
         mel=out[0], mel_post=out[1], gate=out[2], align=out[3],
         bn0_running_mean=sd_after["encoder.convolutions.0.1.running_mean"],
         bn0_running_var=sd_after["encoder.convolutions.0.1.running_var"])


def grad_sample_index(name, numel, n=96):
    """Deterministic flat indices at which the gradient of parameter `name` is stored in the fixture."""
    h = 0
    for ch in name:
        h = (h * 131 + ord(ch)) % 2147483647
    g = torch.Generator().manual_seed(h)
    return torch.randint(0, numel, (min(n, numel),), generator=g)


def gate_targets(ol, T_mel):
    """data_utils.py:105-107: gate_padded[i, len_i - 1:] = 1."""
    gt = torch.zeros(len(ol), T_mel)
    for i, n in enumerate(ol.tolist()):
        gt[i, n - 1:] = 1.0
    return gt


def grad_case(name, training, B, T_text, T_mel, wseed, seed, wscale=2.0, n_samples=96, keep_outputs=True,
              ref64=False):
    """Full training step of the REFERENCE (forward + Tacotron2Loss + backward, autograd) with injected dropout
    masks; the fixture keeps the loss and, per parameter, sum / abs-sum / max of the gradient plus 96 sampled entries."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_loss_function", os.path.join(REFERENCE_DIR, "loss_function.py"))
    lf = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(lf)
    sd = synth_state_dict(wseed, scale=wscale)
    g = torch.Generator().manual_seed(seed)
    text = rand_text(B, T_text, seed + 1)
    tl = torch.sort(torch.randint(T_text // 3, T_text + 1, (B,), generator=g), descending=True)[0]
    tl[0] = T_text
    ol = torch.randint(T_mel // 3, T_mel + 1, (B,), generator=g); ol[1] = T_mel
    mels = torch.randn(B, 80, T_mel, generator=g)
    for i, n in enumerate(ol.tolist()):
        mels[i, :, n:] = 0.0                                    # TextMelCollate zero-pads (data_utils.py:97-104)
    pk = keep_mask((T_mel + 1, 2, B, 256), 0.5, seed + 2)
    ak = keep_mask((T_mel, B, 1024), 0.1, seed + 3)
    dk = keep_mask((T_mel, B, 1024), 0.1, seed + 4)
    ek = keep_mask((3, B, 512, T_text), 0.5, seed + 5)
    qk4 = keep_mask((4, B, 512, T_mel), 0.5, seed + 6)
    qk1 = keep_mask((B, 80, T_mel), 0.5, seed + 7)
    model = build(sd, training)
    if training:
        masks = [ek[i].bool() for i in range(3)] + [pk[:, 0].bool(), pk[:, 1].bool()]
        for t in range(T_mel):
            masks += [ak[t].bool(), dk[t].bool()]
        masks += [qk4[i].bool() for i in range(4)] + [qk1.bool()]
    else:
        masks = [pk[:, 0].bool(), pk[:, 1].bool()]
    gt = gate_targets(ol, T_mel)
    with injected_dropout(ref, MaskInjector(masks)) as inj:
        out = model((text, tl, mels, int(tl.max()), ol))
        assert inj.calls == len(masks)
    loss = lf.Tacotron2Loss()(out, (mels, gt))
    loss.backward()
    arrays = dict(training=int(training), B=B, T_text=T_text, T_mel=T_mel, wseed=wseed, seed=seed, wscale=wscale,
                  wsum=weights_checksum(sd), text_lengths=tl, output_lengths=ol, mels_in=mels, gate_target=gt,
                  loss=loss.detach(), mel=out[0].detach(), mel_post=out[1].detach(), n_samples=n_samples)
    if not keep_outputs:      # full-size case: the inputs are regenerated from the seeds, outputs sub-sampled in time
        idx = torch.tensor(full_frame_index(T_mel, 2 * FULL_STRIDE))
        arrays.update(mel=out[0].detach()[:, :, idx], mel_post=out[1].detach()[:, :, idx], frame_index=idx, gate=out[2].detach())
        del arrays["mels_in"], arrays["gate_target"]
    for k, p_ in model.named_parameters():
        gr = p_.grad.detach().double().reshape(-1)
        idx = grad_sample_index(k, gr.numel(), n_samples)
        arrays["g/" + k] = torch.cat((torch.stack((gr.sum(), gr.abs().sum(), gr.abs().max())), gr[idx]))
    if ref64:
        # The same step through the reference in DOUBLE precision (model.double()): at B=64 / T_mel=800 the reference's
        # fp32 autograd is itself 1e-3 ... 1e-2 (relative to the gradient's maximum) away from this for the parameters
        # behind the training-mode BatchNorms (DESIGN.md section 2), so the fp64 values are what an fp32-grade
        # implementation is held to, with the fp32 reference's own deviation as the yardstick.
        model64 = build(sd, training).double()
        with injected_dropout(ref, MaskInjector(masks)) as inj:
            out64 = model64((text, tl, mels.double(), int(tl.max()), ol))
        loss64 = lf.Tacotron2Loss()(out64, (mels.double(), gt.double()))
        loss64.backward()
        arrays["loss64"] = loss64.detach()
        worst = {}
        for k, p_ in model64.named_parameters():
            gr = p_.grad.detach().reshape(-1)
            idx = grad_sample_index(k, gr.numel(), n_samples)
            arrays["g64/" + k] = torch.cat((torch.stack((gr.sum(), gr.abs().sum(), gr.abs().max())), gr[idx]))
            gmax = float(gr.abs().max())
            if gmax > 1e-5:
                worst[k] = float((torch.as_tensor(arrays["g/" + k])[3:] - gr[idx]).abs().max()) / gmax
        top = sorted(worst.items(), key=lambda kv: -kv[1])[:8]
        print(name, "fp32 reference vs fp64 reference, largest sampled deviations / max|g|:",
              ", ".join("%s %.1e" % kv for kv in top))
    print(name, "loss", float(loss))
    save(name, **arrays)


def import_reference_stft():
    """The reference's stft.py with functional stand-ins for the two librosa.util helpers it imports (librosa itself is
    not in this image): pad_center = symmetric zero padding, tiny = smallest normal float32."""
    import importlib.util
    import types

    def pad_center(data, size, axis=-1, **kw):
        n = data.shape[axis]
        lpad = int((size - n) // 2)
        lengths = [(0, 0)] * data.ndim
        lengths[axis] = (lpad, int(size - n - lpad))
        return np.pad(data, lengths, mode="constant")
    saved = {k: sys.modules.get(k) for k in ("librosa", "librosa.util", "librosa.filters", "audio_processing", "stft")}
    lib, lu, lf = types.ModuleType("librosa"), types.ModuleType("librosa.util"), types.ModuleType("librosa.filters")
    lu.pad_center, lu.tiny, lf.mel = pad_center, (lambda x: np.finfo(np.float32).tiny), None
    lib.util, lib.filters = lu, lf
    sys.modules.update({"librosa": lib, "librosa.util": lu, "librosa.filters": lf})
    sys.path.insert(0, REFERENCE_DIR)
    try:
        spec = importlib.util.spec_from_file_location("t2_reference_stft", os.path.join(REFERENCE_DIR, "stft.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        sys.path.remove(REFERENCE_DIR)
        for k, v in saved.items():
            sys.modules.pop(k, None)
            if v is not None:
                sys.modules[k] = v
    return mod


STFT_SETTINGS = ((1024, 256, 1024), (800, 200, 800), (512, 128, 400))     # (filter_length, hop_length, win_length)


def stft_settings_case():
    """The reference's stft.STFT for three filter / hop / window settings on seeded 2-row signals: the magnitudes, and 4096
    seeded samples plus the absolute sum of the windowed Fourier basis (the whole basis is 4 MB at filter_length 1024)."""
    mod = import_reference_stft()
    g = torch.Generator().manual_seed(0)
    out = {}
    for fl, hop, win in STFT_SETTINGS:
        ref_stft = mod.STFT(fl, hop, win)
        basis = ref_stft.forward_basis[:, 0, :].reshape(-1)
        idx = torch.randint(0, basis.numel(), (4096,), generator=g)
        mag, _ = ref_stft.transform(stft_inputs(seed=fl, n=5000))
        out.update({"mag_%d" % fl: mag, "basis_index_%d" % fl: idx.to(torch.int32), "basis_%d" % fl: basis[idx],
                    "basis_abs_sum_%d" % fl: basis.double().abs().sum()})
    save("stft_mag_settings", **out)


def import_reference_collate():
    """The reference's data_utils.py with stand-ins for the modules it imports but TextMelCollate does not use."""
    import importlib.util
    import types
    saved = {k: sys.modules.get(k) for k in ("layers", "utils", "text")}
    try:
        for k in saved:
            sys.modules[k] = types.ModuleType(k)
        sys.modules["utils"].load_wav_to_torch = sys.modules["utils"].load_filepaths_and_text = None
        sys.modules["text"].text_to_sequence = None
        spec = importlib.util.spec_from_file_location("t2_reference_data_utils", os.path.join(REFERENCE_DIR, "data_utils.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            sys.modules.pop(k, None)
            if v is not None:
                sys.modules[k] = v
    return mod


def refs_cases():
    """Fixtures for tests/test_oracle_vs_reference.py and the reference checks of tests/test_boundary_cpu.py."""
    # Tacotron2.inference of the reference itself at B=1, 12 steps (its own stop loop, injected prenet masks)
    sd = synth_state_dict(5, gate_bias=-10.0, scale=2.0)
    model = build(sd)
    model.decoder.max_decoder_steps = 12
    text, keep = rand_text(1, 19, 3), keep_mask((12, 2, 1, 256), 0.5, 4)
    masks = [keep[t, l].bool() for t in range(12) for l in range(2)]
    with torch.no_grad(), injected_dropout(ref, MaskInjector(masks)):
        r = model.inference(text)
    save("ref_inference_b1_t19", wsum=weights_checksum(sd), mel=r[0], mel_post=r[1], gate=r[2], align=r[3])
    # state_dict keys / shapes, and the initial weights under torch.manual_seed(1234) as one digest per entry
    torch.manual_seed(1234)
    sd = ref.Tacotron2(default_hparams()).state_dict()
    save("ref_init_seed1234", keys=np.array(list(sd)), shapes=np.array([",".join(map(str, v.shape)) for v in sd.values()]),
         digests=np.array([tensor_digest(v) for v in sd.values()]))
    # a whole training step (forward + Tacotron2Loss + backward) of the reference
    grad_case("grad_train_b3_t15_m8", True, 3, 15, 8, 4321, 91, n_samples=512)
    stft_settings_case()
    # TextMelCollate on the batches of tests.common.collate_batches: digests of its five outputs
    coll = import_reference_collate()
    fixed, trials = collate_batches()
    save("ref_collate", digests=np.array([[[tensor_digest(t) for t in coll.TextMelCollate(nfs)(b)] for b in [fixed] + trials[nfs]]
                                          for nfs in (1, 2)]))


def stft_case():
    """STFT magnitudes of the reference's own stft.STFT(1024, 256, 1024) (stft.py:69-94) for a seeded 2-row signal."""
    mod = import_reference_stft()
    ref_stft = mod.STFT(1024, 256, 1024)
    y = stft_inputs()
    mag, _ = ref_stft.transform(y)
    save("stft_mag", y=y, mag=mag, basis_abs_sum=ref_stft.forward_basis.double().abs().sum())


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "stft":
        stft_case()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "full":        # the configurations the benchmark numbers are quoted on
        which = sys.argv[2:] or ["infer64", "infer32", "grad64"]
        if "infer64" in which:   # BASELINE.json configs[1]: B=64, T_text=150, 800 steps, the bench weights (scale 1.0)
            full_infer_case("full_infer_b64_t150_s800", 64, 150, 800, 1234, 101, 102, 1.0)
        if "infer32" in which:   # configs[4] per GPU: B=32, T_text=300, 2000 steps
            full_infer_case("full_infer_b32_t300_s2000", 32, 300, 2000, 1234, 111, 112, 1.0)
        if "grad64" in which:    # configs[2]: teacher-forced training step B=64, T_mel=800
            grad_case("full_grad_train_b64_t150_m800", True, 64, 150, 800, 1234, 160, wscale=1.0, n_samples=1024,
                      keep_outputs=False, ref64=True)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "refs":
        refs_cases()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "grads":
        grad_case("grad_train_b4", True, 4, 24, 12, 1234, 60)
        grad_case("grad_eval_b3", False, 3, 17, 9, 77, 70)
        sys.exit(0)
    infer_case("infer_b1_t50", 1, 50, 40, 0.95, 1234, 11, 12)
    infer_case("infer_b4_t24", 4, 24, 32, 0.93, 1234, 21, 22)
    infer_case("infer_b3_t37", 3, 37, 16, 0.90, 77, 31, 32, wscale=1.0)
    forward_case("forward_train_b4", True, 4, 24, 12, 1234, 40)
    forward_case("forward_eval_b4", False, 4, 24, 12, 1234, 50)
