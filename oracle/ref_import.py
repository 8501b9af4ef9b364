"""TEST INFRASTRUCTURE ONLY -- never imported by the product path.

Imports the *unmodified* reference ``model.py`` from a checkout of NVIDIA/tacotron2
named by ``T2_REFERENCE_DIR`` so that golden vectors can be generated for
``tests/golden`` (``tools/make_golden.py``); those fixtures are what pin the CPU
restatement in ``oracle/tacotron2_oracle.py`` and the CUDA path.  No test imports it.

Four non-invasive shims (SURVEY.md section 8(c)):
  1. stub ``librosa`` (layers.py:2, stft.py:38, audio_processing.py:4 import it; it is
     never reached from model.py),
  2. a TF-free hparams namespace with the defaults of hparams.py:12-85,
  3. ``model.get_mask_from_lengths`` rebound to a device-agnostic version
     (utils.py:8 hard-codes torch.cuda.LongTensor),
  4. ``model.F.dropout`` optionally rebound to a mask-injecting dropout so both
     sides of a parity test consume the same Bernoulli masks.
"""
import os
import sys
import types
from types import SimpleNamespace

REFERENCE_DIR = os.environ.get("T2_REFERENCE_DIR", "")


def reference_available():
    return bool(REFERENCE_DIR) and os.path.isfile(os.path.join(REFERENCE_DIR, "model.py"))


def default_hparams(**overrides):
    """Defaults of hparams.py:12-85 (n_symbols = 148, text/symbols.py:9-18)."""
    hp = dict(
        epochs=500, iters_per_checkpoint=1000, seed=1234, dynamic_loss_scaling=True,
        fp16_run=False, distributed_run=False, dist_backend="nccl",
        dist_url="tcp://localhost:54321", cudnn_enabled=True, cudnn_benchmark=False,
        ignore_layers=['embedding.weight'],
        load_mel_from_disk=False, text_cleaners=['english_cleaners'],
        max_wav_value=32768.0, sampling_rate=22050, filter_length=1024, hop_length=256,
        win_length=1024, n_mel_channels=80, mel_fmin=0.0, mel_fmax=8000.0,
        n_symbols=148, symbols_embedding_dim=512,
        encoder_kernel_size=5, encoder_n_convolutions=3, encoder_embedding_dim=512,
        n_frames_per_step=1, decoder_rnn_dim=1024, prenet_dim=256,
        max_decoder_steps=1000, gate_threshold=0.5, p_attention_dropout=0.1,
        p_decoder_dropout=0.1, attention_rnn_dim=1024, attention_dim=128,
        attention_location_n_filters=32, attention_location_kernel_size=31,
        postnet_embedding_dim=512, postnet_kernel_size=5, postnet_n_convolutions=5,
        use_saved_learning_rate=False, learning_rate=1e-3, weight_decay=1e-6,
        grad_clip_thresh=1.0, batch_size=64, mask_padding=True)
    hp.update(overrides)
    return SimpleNamespace(**hp)


_ref_model = None


def import_reference_model():
    """Returns the reference ``model`` module (cached)."""
    global _ref_model
    if _ref_model is not None:
        return _ref_model
    if not reference_available():
        raise RuntimeError("no reference checkout at T2_REFERENCE_DIR=%r" % REFERENCE_DIR)
    for name in ("librosa", "librosa.filters", "librosa.util"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.mel = lambda *a, **k: None
            m.normalize = lambda *a, **k: None
            m.pad_center = lambda *a, **k: None
            m.tiny = lambda *a, **k: 1e-30
            sys.modules[name] = m
    sys.modules["librosa"].filters = sys.modules["librosa.filters"]
    sys.modules["librosa"].util = sys.modules["librosa.util"]
    import importlib.util
    saved_path = list(sys.path)
    saved_mods = {k: sys.modules.get(k) for k in ("model", "layers", "utils", "stft",
                                                   "audio_processing")}
    try:
        sys.path.insert(0, REFERENCE_DIR)
        for k in saved_mods:
            sys.modules.pop(k, None)
        spec = importlib.util.spec_from_file_location(
            "t2_reference_model", os.path.join(REFERENCE_DIR, "model.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        sys.path[:] = saved_path
        for k, v in saved_mods.items():
            sys.modules.pop(k, None)
            if v is not None:
                sys.modules[k] = v
    import torch

    def get_mask_from_lengths(lengths):  # shim 3 (utils.py:6-10 semantics)
        max_len = int(torch.max(lengths).item())
        ids = torch.arange(0, max_len, device=lengths.device, dtype=torch.long)
        return (ids < lengths.unsqueeze(1)).bool()

    mod.get_mask_from_lengths = get_mask_from_lengths
    mod._orig_dropout = mod.F.dropout
    _ref_model = mod
    return mod


class MaskInjector:
    """Shim 4: a stand-in for ``F.dropout`` that consumes caller-supplied keep-masks.

    ``masks`` is a list; every dropout call with ``training=True`` and p>0 pops the next
    entry (a uint8/bool keep mask of the input's shape) and returns x*mask/(1-p), which is
    what F.dropout computes for the same Bernoulli draw.
    """

    def __init__(self, masks):
        self.masks = list(masks)
        self.calls = 0

    def __call__(self, x, p=0.5, training=True, inplace=False):
        if not training or p == 0.0:
            return x
        m = self.masks[self.calls]
        self.calls += 1
        assert tuple(m.shape) == tuple(x.shape), (m.shape, x.shape)
        return x * m.to(x.dtype) * (1.0 / (1.0 - p))


class injected_dropout:
    """Context manager rebinding the reference module's F.dropout (shared torch.nn.functional
    attribute is NOT touched: the reference does ``from torch.nn import functional as F`` so we
    swap the module-level name ``F`` for a proxy)."""

    def __init__(self, ref_mod, injector):
        self.ref_mod, self.injector = ref_mod, injector

    def __enter__(self):
        import torch.nn.functional as realF
        proxy = types.SimpleNamespace(**{k: getattr(realF, k) for k in dir(realF)
                                         if not k.startswith("__")})
        proxy.dropout = self.injector
        self._saved = self.ref_mod.F
        self.ref_mod.F = proxy
        return self.injector

    def __exit__(self, *exc):
        self.ref_mod.F = self._saved
        return False
