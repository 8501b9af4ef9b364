"""Shared helpers for the test-suite: deterministic synthetic weights / inputs / dropout masks.

Everything is generated from ``torch.Generator`` CPU seeds so the build container (where the
golden vectors are produced from the reference) and the GPU box (same image) agree bit for bit;
each golden file also stores a checksum of the weights it was produced with.
"""
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")

# name -> shape for the 84 state_dict entries of the default hparams (SURVEY.md section 8(b1))
def state_dict_shapes():
    s = {"embedding.weight": (148, 512)}
    for i in range(3):
        p = "encoder.convolutions.%d." % i
        s[p + "0.conv.weight"] = (512, 512, 5); s[p + "0.conv.bias"] = (512,)
        for n in ("weight", "bias", "running_mean", "running_var"):
            s[p + "1." + n] = (512,)
        s[p + "1.num_batches_tracked"] = ()
    for suf in ("", "_reverse"):
        s["encoder.lstm.weight_ih_l0" + suf] = (1024, 512)
        s["encoder.lstm.weight_hh_l0" + suf] = (1024, 256)
        s["encoder.lstm.bias_ih_l0" + suf] = (1024,)
        s["encoder.lstm.bias_hh_l0" + suf] = (1024,)
    d = "decoder."
    s[d + "prenet.layers.0.linear_layer.weight"] = (256, 80)
    s[d + "prenet.layers.1.linear_layer.weight"] = (256, 256)
    s[d + "attention_rnn.weight_ih"] = (4096, 768); s[d + "attention_rnn.weight_hh"] = (4096, 1024)
    s[d + "attention_rnn.bias_ih"] = (4096,); s[d + "attention_rnn.bias_hh"] = (4096,)
    a = d + "attention_layer."
    s[a + "query_layer.linear_layer.weight"] = (128, 1024)
    s[a + "memory_layer.linear_layer.weight"] = (128, 512)
    s[a + "v.linear_layer.weight"] = (1, 128)
    s[a + "location_layer.location_conv.conv.weight"] = (32, 2, 31)
    s[a + "location_layer.location_dense.linear_layer.weight"] = (128, 32)
    s[d + "decoder_rnn.weight_ih"] = (4096, 1536); s[d + "decoder_rnn.weight_hh"] = (4096, 1024)
    s[d + "decoder_rnn.bias_ih"] = (4096,); s[d + "decoder_rnn.bias_hh"] = (4096,)
    s[d + "linear_projection.linear_layer.weight"] = (80, 1536)
    s[d + "linear_projection.linear_layer.bias"] = (80,)
    s[d + "gate_layer.linear_layer.weight"] = (1, 1536)
    s[d + "gate_layer.linear_layer.bias"] = (1,)
    chans = [(512, 80), (512, 512), (512, 512), (512, 512), (80, 512)]
    for i, (co, ci) in enumerate(chans):
        p = "postnet.convolutions.%d." % i
        s[p + "0.conv.weight"] = (co, ci, 5); s[p + "0.conv.bias"] = (co,)
        for n in ("weight", "bias", "running_mean", "running_var"):
            s[p + "1." + n] = (co,)
        s[p + "1.num_batches_tracked"] = ()
    return s


def synth_state_dict(seed=1234, gate_bias=None, scale=1.0, gate_sign=1.0):
    """Deterministic weights with magnitudes like the reference's initialisation (Xavier-style
    bounds for matrices, U(+-1/sqrt(H)) for LSTMs) and NON-trivial BatchNorm statistics so the
    BN folding is exercised."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for name, shape in state_dict_shapes().items():
        if name.endswith("num_batches_tracked"):
            sd[name] = torch.tensor(0, dtype=torch.long)
        elif name.endswith("running_var"):
            sd[name] = torch.rand(shape, generator=g) + 0.5
        elif name.endswith("running_mean"):
            sd[name] = torch.randn(shape, generator=g) * 0.1
        elif ".1.weight" in name:                      # BN gamma
            sd[name] = torch.rand(shape, generator=g) + 0.5
        elif ".1.bias" in name:                        # BN beta
            sd[name] = torch.randn(shape, generator=g) * 0.1
        elif "lstm" in name or "_rnn." in name:
            H = 256 if "encoder" in name else 1024
            sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * (scale / math.sqrt(H))
        elif len(shape) >= 2:
            fan_out = shape[0] * (shape[2] if len(shape) == 3 else 1)
            fan_in = shape[1] * (shape[2] if len(shape) == 3 else 1)
            bound = scale * math.sqrt(6.0 / (fan_in + fan_out))
            if name == "embedding.weight":
                bound = math.sqrt(3.0) * math.sqrt(2.0 / (148 + 512))
            sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * bound
        else:                                          # biases
            sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * 0.05
    if gate_bias is not None:
        sd["decoder.gate_layer.linear_layer.bias"] = torch.tensor([float(gate_bias)])
    sd["decoder.gate_layer.linear_layer.weight"] = sd["decoder.gate_layer.linear_layer.weight"] * gate_sign
    return sd


def weights_checksum(sd):
    tot = 0.0
    for k in sorted(sd):
        if sd[k].dtype.is_floating_point:
            tot += float(sd[k].double().abs().sum())
    return tot


def keep_mask(shape, p_drop, seed):
    """uint8 Bernoulli keep-mask (1 = keep), P(keep) = 1 - p_drop."""
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(shape, generator=g) >= p_drop).to(torch.uint8)


def rand_text(B, T, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 148, (B, T), generator=g)


def rel_err(a, b):
    """max |a-b| / max |b|  -- the 'relative fp32' measure used for the 1e-3 parity bar."""
    a = a.detach().double().cpu(); b = b.detach().double().cpu()
    den = float(b.abs().max())
    return float((a - b).abs().max()) / (den if den > 0 else 1.0)


def tensor_digest(t):
    """SHA-256 of a tensor's dtype, shape and bytes: equal digests <=> torch.equal with the same dtype.  Lets a fixture pin
    large exact outputs (initial weights, collated batches) in a few bytes."""
    import hashlib
    t = t.detach().cpu().contiguous()
    h = hashlib.sha256(("%s %s " % (t.dtype, tuple(t.shape))).encode())
    h.update(t.numpy().tobytes())
    return h.hexdigest()


def stft_inputs(seed=0, n=6000):
    """Two seeded test signals in [-1, 1]: two sines plus noise, and clipped noise."""
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(n) / 22050.0
    return torch.stack([0.3 * torch.sin(2 * math.pi * 220 * t) + 0.2 * torch.sin(2 * math.pi * 1870 * t) + 0.05 * torch.randn(n, generator=g),
                        (0.5 * torch.randn(n, generator=g)).clamp(-1, 1)])


def collate_batches(n_trials=20):
    """Ragged (text, mel) batches for TextMelCollate: a fixed batch of five, then for n_frames_per_step = 1 and 2 in turn
    `n_trials` random batches (ties in the text lengths included).  Returns (fixed, {1: [...], 2: [...]})."""
    g = torch.Generator().manual_seed(0)
    fixed = [(torch.randint(1, 148, (n_text,), generator=g), torch.randn(80, n_mel, generator=g))
             for n_text, n_mel in [(7, 13), (12, 5), (3, 21), (12, 9), (1, 1)]]
    trials = {}
    for nfs in (1, 2):
        trials[nfs] = []
        for _ in range(n_trials):
            n = int(torch.randint(1, 9, (1,), generator=g))
            trials[nfs].append([(torch.randint(1, 148, (int(torch.randint(1, 12, (1,), generator=g)),), generator=g),
                                 torch.randn(80, int(torch.randint(1, 30, (1,), generator=g)), generator=g)) for _ in range(n)])
    return fixed, trials
