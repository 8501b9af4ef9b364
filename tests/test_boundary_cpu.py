"""CPU: the drop-in boundary -- nn.Module surface (state_dict keys / shapes / initialisation),
TF-free hparams, the C-ABI library loads and exports every symbol include/t2b200.h declares, the
ctypes structs match the C layout, and the product path fails loudly without CUDA tensors."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest
import torch

import tacotron2_b200 as t2
from tacotron2_b200 import _capi
from tacotron2_b200._engine import weight_table_spec
from tests.common import GOLDEN_DIR, ROOT, collate_batches, state_dict_shapes, synth_state_dict, tensor_digest


def _ensure_built():
    if not os.path.isfile(_capi.LIB_PATH):
        import __graft_entry__ as g
        g.build()


def test_state_dict_layout_matches_reference_table():
    model = t2.Tacotron2(t2.create_hparams())
    sd = model.state_dict()
    want = state_dict_shapes()
    assert list(sd.keys()) == list(want.keys())
    assert len(sd) == 84
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(want[k]), k
    spec = weight_table_spec(t2.create_hparams())
    assert [n for n, _ in spec] == list(want.keys())
    assert sum(p.numel() for p in model.parameters()) == 28193153       # SURVEY.md section 2.1


def test_same_seed_same_init_as_reference():
    """Under torch.manual_seed(1234) every state_dict entry is bit-identical to the reference's initialisation (one
    digest per entry in tests/golden/ref_init_seed1234.npz)."""
    g = np.load(os.path.join(GOLDEN_DIR, "ref_init_seed1234.npz"))
    torch.manual_seed(1234)
    b = t2.Tacotron2(t2.create_hparams()).state_dict()
    assert list(b) == g["keys"].tolist()
    for k, d in zip(g["keys"].tolist(), g["digests"].tolist()):
        assert tensor_digest(b[k]) == d, k


def test_load_state_dict_roundtrip_and_attributes():
    model = t2.Tacotron2(t2.create_hparams())
    sd = synth_state_dict(3)
    model.load_state_dict(sd)
    for k, v in model.state_dict().items():
        assert torch.equal(v, sd[k])
    # attributes callers poke from outside (train.py:76, inference.ipynb)
    model.decoder.attention_layer.score_mask_value = -65504.0
    model.decoder.max_decoder_steps = 7
    model.decoder.gate_threshold = 0.4
    assert model.decoder.attention_layer.score_mask_value == -65504.0
    assert model.eval() is model and model.train() is model
    fired = []
    model.register_forward_hook(lambda *a: fired.append(1))   # distributed.py:169-172 relies on this


def test_hparams_defaults_and_parse():
    hp = t2.create_hparams("batch_size=8,fp16_run=True,learning_rate=0.01")
    assert hp.batch_size == 8 and hp.fp16_run is True and abs(hp.learning_rate - 0.01) < 1e-12
    assert hp.n_symbols == 148 and hp.max_decoder_steps == 1000 and hp.mask_padding is True
    with pytest.raises(ValueError):
        t2.create_hparams("no_such=1")


def test_product_path_needs_cuda():
    model = t2.Tacotron2(t2.create_hparams()).eval()
    with torch.no_grad(), pytest.raises(RuntimeError, match="CUDA"):
        model.inference(torch.zeros(1, 5, dtype=torch.long))


def test_library_exports_every_declared_symbol():
    _ensure_built()
    header = open(os.path.join(ROOT, "include", "t2b200.h")).read()
    declared = set(re.findall(r"\b(t2_[a-z0-9_]+)\s*\(", header))
    selftests = {n for n in declared if n.startswith("t2_selftest_")}      # declared under #ifdef T2_SELFTEST
    assert selftests == set(_capi.SELFTEST_EXPORTS), selftests ^ set(_capi.SELFTEST_EXPORTS)
    assert declared - selftests == set(_capi.EXPORTS), (declared - selftests) ^ set(_capi.EXPORTS)
    L = _capi.lib()
    for name in declared - selftests:
        assert hasattr(L, name), name
    for name in selftests:                 # the product library carries no self-test / micro-benchmark code ...
        assert not hasattr(L, name), name
    S = _capi.selftest_lib()               # ... the self-test build of the same sources does
    for name in declared:
        assert hasattr(S, name), name
    assert L.t2_abi_version() == 1


def test_ctypes_structs_match_c_layout(tmp_path):
    """sizeof/offsetof of every args struct as gcc sees the header == the ctypes mirror."""
    src = tmp_path / "layout.c"
    fields = {
        "T2Config": ["n_mel_channels", "postnet_n_convolutions", "p_attention_dropout", "bn_eps"],
        "T2EncoderArgs": ["text", "embedded", "lengths", "B", "T", "training", "keep", "seed", "memory", "ws", "ws_bytes",
                          "stash", "stash_bytes"],
        "T2EncoderBwdArgs": ["text", "embedded", "lengths", "B", "T", "training", "keep", "seed", "stash", "stash_bytes",
                             "d_memory", "d_embedded", "grads", "n_grads", "ws", "ws_bytes"],
        "T2PostnetBwdArgs": ["B", "T", "training", "add_residual", "keep", "seed", "wgrad_lengths", "stash", "stash_bytes",
                             "d_mel_post", "d_mel", "grads", "n_grads", "ws", "ws_bytes"],
        "T2DecoderArgs": ["mode", "impl", "training", "memory", "memory_lengths", "B", "T_enc", "n_steps_cap",
                          "teacher_prenet", "prenet_keep", "att_keep", "dec_keep", "seed", "gate_threshold",
                          "score_mask_value", "mel", "gate", "align", "mel_lengths", "n_steps", "ws", "ws_bytes",
                          "stash", "stash_bytes"],
        "T2DecoderBwdArgs": ["memory", "memory_lengths", "B", "T_enc", "T_mel", "training", "teacher_prenet", "att_keep",
                             "dec_keep", "seed", "score_mask_value", "align", "stash", "stash_bytes", "d_mel", "d_gate",
                             "d_align", "d_memory", "d_prenet", "grads", "n_grads", "ws", "ws_bytes"],
        "T2PrenetBwdArgs": ["frames", "M", "keep", "seed", "d_out", "grads", "n_grads", "ws", "ws_bytes"],
        "T2AdamArgs": ["n", "params", "grads", "exp_avg", "exp_avg_sq", "numel", "lr", "beta1", "beta2", "eps", "weight_decay",
                       "max_norm", "step", "grad_norm", "ws", "ws_bytes"],
        "T2PostnetArgs": ["mel", "mel_batch_stride", "lengths", "B", "T", "training", "keep", "seed",
                          "add_residual", "mel_post", "ws", "ws_bytes", "stash", "stash_bytes"],
        "T2AmpAdamArgs": ["n", "model_params", "param_is_half", "grads", "grad_is_half", "master", "exp_avg", "exp_avg_sq", "numel",
                          "lr", "beta1", "beta2", "eps", "weight_decay", "max_norm", "growth_interval", "growth_factor",
                          "backoff_factor", "state", "grad_norm", "skipped", "ws", "ws_bytes"],
        "T2LossArgs": ["mel", "mel_post", "gate", "mel_target", "gate_target", "output_lengths", "B", "C", "T", "loss", "d_mel",
                       "d_mel_post", "d_gate", "ws", "ws_bytes"],
        "T2MelSpecArgs": ["y", "B", "n_samples", "filter_length", "hop_length", "n_mel", "forward_basis", "mel_basis", "clip_val",
                          "mel", "ws", "ws_bytes"],
        "T2CollateArgs": ["text_flat", "text_offsets", "mel_flat", "mel_offsets", "B", "n_mel", "T_max", "L_pad", "order",
                          "text_padded", "input_lengths", "mel_padded", "gate_padded", "output_lengths"],
    }
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "t2b200.h"', 'int main(void){']
    for s, fs in fields.items():
        lines.append('printf("%s %%zu\\n", sizeof(%s));' % (s, s))
        for f in fs:
            lines.append('printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (s, f, s, f))
    lines.append('return 0;}')
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = dict(l.split() for l in subprocess.check_output([str(exe)]).decode().splitlines())
    for s, fs in fields.items():
        cls = getattr(_capi, s)
        assert int(out[s]) == ctypes.sizeof(cls), s
        for f in fs:
            assert int(out["%s.%s" % (s, f)]) == getattr(cls, f).offset, (s, f)


def test_text_mel_collate_matches_reference_semantics():
    """tacotron2_b200.data_utils.TextMelCollate vs its documented properties and vs the outputs of the reference's collate
    function (data_utils.py:67-111) on the same batches (digests in tests/golden/ref_collate.npz)."""
    from tacotron2_b200.data_utils import TextMelCollate
    batch, trials = collate_batches()
    ref = np.load(os.path.join(GOLDEN_DIR, "ref_collate.npz"))["digests"]
    for j, nfs in enumerate((1, 2)):
        out = TextMelCollate(nfs)(batch)
        text, tl, mel, gate, ol = out
        assert tl.tolist() == sorted(tl.tolist(), reverse=True) and mel.shape[2] % nfs == 0 and mel.shape[2] >= int(ol.max())
        for i in range(len(batch)):
            assert int((text[i] != 0).sum()) == int(tl[i]) and bool((mel[i, :, int(ol[i]):] == 0).all())
            assert gate[i].tolist() == [0.0] * (int(ol[i]) - 1) + [1.0] * (mel.shape[2] - int(ol[i]) + 1)
        assert [tensor_digest(a) for a in out] == ref[j, 0].tolist()
        for trial, rb in enumerate(trials[nfs]):     # random ragged batches (ties in the text lengths included)
            assert [tensor_digest(a) for a in TextMelCollate(nfs)(rb)] == ref[j, 1 + trial].tolist(), trial


def test_parse_batch_returns_the_reference_structure():
    """Tacotron2.parse_batch (model.py:473-485) on a collated batch: ((text, input_lengths, mel, max_len, output_lengths),
    (mel, gate)); on a CPU-only host to_gpu() leaves the tensors where they are."""
    from tacotron2_b200.data_utils import TextMelCollate
    g = torch.Generator().manual_seed(1)
    batch = [(torch.randint(1, 148, (n,), generator=g), torch.randn(80, m, generator=g)) for n, m in [(4, 6), (9, 3), (2, 8)]]
    model = t2.Tacotron2(t2.create_hparams())
    x, y = model.parse_batch(TextMelCollate(1)(batch))
    assert len(x) == 5 and len(y) == 2 and x[3] == 9 and x[0].dtype == torch.int64 and x[2].dtype == torch.float32
    assert x[1].tolist() == [9, 4, 2] and x[4].tolist() == [3, 6, 8] and torch.equal(x[2], y[0]) and y[1].shape == (3, 8)


def test_deepcopy_and_pickle_resolve_their_own_root():
    """copy.deepcopy(model) / torch.save(model): the weak back-references and the engine are per-instance runtime state
    (ADVICE r1: a copy's children used to resolve the ORIGINAL model's engine and parameters)."""
    import copy
    import io
    model = t2.Tacotron2(t2.create_hparams())
    model._t2_link()
    assert model.decoder._t2_root() is model and model.decoder.prenet._t2_root() is model
    clone = copy.deepcopy(model)
    clone._t2_link()
    for child in (clone.encoder, clone.decoder, clone.postnet, clone.decoder.prenet):
        assert child._t2_root() is clone
    assert model.decoder._t2_root() is model                      # the original is untouched
    assert "_t2_engine_obj" not in clone.__dict__
    with torch.no_grad():
        clone.decoder.gate_layer.linear_layer.bias.fill_(3.0)
    assert float(model.decoder.gate_layer.linear_layer.bias) != 3.0
    buf = io.BytesIO()
    torch.save(model, buf)                                        # used to raise "cannot pickle weakref"
    buf.seek(0)
    loaded = torch.load(buf, weights_only=False)
    loaded._t2_link()
    assert loaded.decoder._t2_root() is loaded
    assert all(torch.equal(a, b) for a, b in zip(loaded.state_dict().values(), model.state_dict().values()))
    # a stand-alone Decoder owns its prenet
    dec = copy.deepcopy(t2.Decoder(t2.create_hparams()))
    dec._t2_link()
    assert dec.prenet._t2_root() is dec


def test_engine_cache_key_and_invalidation():
    """The packed device copies are keyed on (generation, pointer, torch version counter, dtype); writes through .data do
    not move the version counter, so there is a public invalidation hook, and load_state_dict calls it (ADVICE r1)."""
    from tacotron2_b200 import _engine
    p = torch.nn.Parameter(torch.ones(4))
    v0 = p._version
    p.data.mul_(2.0)
    assert p._version == v0                                       # the hazard the hook exists for
    g0 = _engine._weights_generation[0]
    t2.invalidate_weights()
    assert _engine._weights_generation[0] == g0 + 1
    eng = _engine.Engine(t2.create_hparams())
    eng.key = ("something",)
    eng.invalidate()
    assert eng.key is None
    model = t2.Tacotron2(t2.create_hparams())
    model.__dict__["_t2_engine_obj"] = eng
    eng.key = ("something",)
    model.load_state_dict(model.state_dict())
    assert eng.key is None
    eng.key = ("something",)
    model.decoder.invalidate_weights()                            # through a child
    assert eng.key is None


def test_bench_roofline_traffic_is_keyed_to_the_kernel_source(tmp_path, monkeypatch):
    """bench.py takes roofline.traffic from profiles/decoder_traffic.json only while decoder_persistent.cu still hashes to the
    captured source; anything else gives None (never a stale literal)."""
    import hashlib
    import json
    import bench
    src = open(os.path.join(ROOT, "tacotron2_b200", "csrc", "decoder_persistent.cu"), "rb").read()
    rec = json.load(open(os.path.join(ROOT, "profiles", "decoder_traffic.json")))
    val, why = bench.decoder_traffic()
    if rec["source_sha16"] == hashlib.sha256(src).hexdigest()[:16]:
        assert val == rec["dram_bytes_per_step"] and val > 1e6
    else:
        assert val is None and "stale" in why
    # a modified source invalidates the record
    fake = tmp_path / "repo"
    (fake / "profiles").mkdir(parents=True)
    (fake / "tacotron2_b200" / "csrc").mkdir(parents=True)
    (fake / "profiles" / "decoder_traffic.json").write_text(json.dumps(rec))
    (fake / "tacotron2_b200" / "csrc" / "decoder_persistent.cu").write_bytes(src + b"\n// edited\n")
    monkeypatch.setattr(bench, "ROOT", str(fake))
    val, why = bench.decoder_traffic()
    assert val is None and "stale" in why
