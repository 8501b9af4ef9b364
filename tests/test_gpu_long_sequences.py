"""GPU (B200): the decoder at long encoder sequences and long teacher-forced runs, where its kernels change code path.

  * the attention energies of the persistent decoder run in rounds of <= 256 positions (decoder_persistent.cu:
    att_rounds = (T + 255) >> 8), and from the second round on the im2col image is a fixed 32 KiB plane;
  * each decoder implementation and the decoder backward accept T_enc only up to a shared-memory limit (below);
  * the time-batched LSTM weight gradients split the T_mel steps into K splits of 100 steps (wgrad_tc.h: wgrad_seg),
    widened by 50 while there would be more than 15 splits, and add the partial sums of the splits at the end.

Every case compares with the CPU oracle on fresh seeded inputs and injected dropout masks.  Inference: 1e-3 of the
maximum, stop decisions bit-exact.  Gradients: the oracle in DOUBLE precision is the truth; every output, every parameter
gradient and d_memory must be within max(1e-3, 4 x the fp32 oracle's own deviation from it) of its maximum."""
import time

import pytest
import torch

import tacotron2_b200 as t2
from oracle import tacotron2_oracle as O
from tacotron2_b200 import _capi
from tests.common import keep_mask, rand_text, rel_err, synth_state_dict
from tests.test_gpu_backward import decoder_case, oracle_decoder_grads
from tests.test_gpu_parity import make_model
from tests.test_oracle_golden import oracle_train_step

pytestmark = pytest.mark.gpu
TOL = 1e-3
SLACK = 4.0

# Largest T_enc each kernel accepts: the largest T whose shared-memory footprint fits its limit.
# decoder_backward.cu, att_bwd_smem(Te) <= 220 KiB:
#   4 * (1712 + 66 * Te4 + 2 * TeP4 + 65 * Te), Te4 = Te rounded up to 4, TeP4 = (Te + 37) & ~3
#   -> 224,192 B at 408, 225,508 B at 409 (limit 225,280)
BWD_MAX_T_ENC = 408
# decoder_persistent.cu, persistent_supported: persistent_smem_bytes(T, 4 stages) <= 227 KiB:
#   183,296 + 8 * ((T + 33) & ~3) + max(8,448, 2,560 * ceil(T / 128))
#   -> 230,144 B at 1664, 232,704 B at 1665 (the 14th 128-position tile; limit 232,448)
PERSISTENT_MAX_T_ENC = 1664
# decoder_stepwise.cu, stepwise_attention_smem(T) <= 200 KiB:
#   4 * (6300 + 35 * T) -> 204,680 B at 1282, 204,820 B at 1283 (limit 204,800)
STEPWISE_MAX_T_ENC = 1282

STEPWISE_TOO_LONG = "too long for the stepwise attention kernel"
PERSISTENT_REFUSED = "does not support this shape"
BWD_TOO_LONG = "too long for the attention kernel"


def fp64(x):
    return x.double() if x is not None and x.dtype == torch.float32 else x


def check_vs_fp64(label, got, r32, r64):
    """got / r32 / r64: name -> tensor.  Error of `got` relative to the fp64 maximum, bar max(TOL, SLACK x the fp32 oracle's
    own error)."""
    errs = {k: rel_err(got[k], r64[k]) for k in r64}
    yard = {k: rel_err(r32[k], r64[k]) for k in r64}
    worst = max(errs, key=errs.get)
    print("%s: worst %.2e (%s; fp32 oracle there %.2e), worst fp32 oracle %.2e" %
          (label, errs[worst], worst, yard[worst], max(yard.values())))
    bad = {k: (errs[k], yard[k]) for k in errs if not errs[k] < max(TOL, SLACK * yard[k])}
    assert not bad, bad


# ---- 1. inference across attention rounds ---------------------------------------------------------------------------
# (B, T_enc, steps, seed, gate_bias).  The gate layer's output feeds nothing but the stop latch, so the bias shifts every
# gate logit of a case by the same amount: the values below stop one row at a live step while the others run on, with
# every live decision at least 1e-2 away from the threshold in the oracle; -10 never stops.
INFER_CASES = [
    (3, 256, 4, 1, -10.0),                        # 1 round
    (3, 257, 4, 2, -0.534),                       # 2 rounds, the second of 1 position; row 1 stops at step 3
    (2, 512, 3, 3, -10.0),                        # 2 full rounds
    (3, 513, 4, 4, -0.965),                       # 3 rounds; row 0 stops at step 3
    (2, 768, 3, 9, -10.0),                        # 3 full rounds
    (2, 769, 3, 5, -10.0),                        # 4 rounds
    (2, STEPWISE_MAX_T_ENC, 3, 6, 0.087),         # row 1 stops at step 2
    (2, STEPWISE_MAX_T_ENC + 1, 3, 7, -10.0),     # the stepwise kernel refuses, the persistent one runs
    (2, PERSISTENT_MAX_T_ENC, 3, 8, 0.169),       # 7 rounds; row 0 stops at step 2
]


@pytest.mark.parametrize("B,T_enc,steps,seed,gate_bias", INFER_CASES)
def test_inference_across_attention_rounds_vs_oracle(B, T_enc, steps, seed, gate_bias):
    t0 = time.time()
    sd = synth_state_dict(200 + seed, gate_bias=gate_bias, scale=2.0)
    text = rand_text(B, T_enc, seed)
    keep = keep_mask((steps, 2, B, 256), 0.5, seed + 50)
    with torch.no_grad():
        ref = O.tacotron2_inference(sd, text, keep, 0.5, steps)
    n = ref[0].shape[2]
    live = torch.arange(n)[None, :] < ref[4][:, None]
    margin = float(ref[2][:, :, 0][live].abs().min())
    assert margin > 5e-3, "stop decisions of this case are ill-posed (gate margin %.1e)" % margin
    impls = [(_capi.IMPL_PERSISTENT, "persistent")]
    if T_enc <= STEPWISE_MAX_T_ENC:
        impls.append((_capi.IMPL_STEPWISE, "stepwise"))
    for impl, name in impls:
        model = make_model(sd, steps, impl)
        with torch.no_grad(), t2.dropout_masks(prenet=keep):
            out = model.inference(text.cuda())
        torch.cuda.synchronize()
        assert model.mel_lengths.cpu().tolist() == ref[4].tolist(), name
        assert out[0].shape == ref[0].shape and out[3].shape == ref[3].shape, name
        errs = [rel_err(a, b) for a, b in zip(out, ref[:4])]
        print("inference [%s] B=%d T_enc=%d: mel %.2e post %.2e gate %.2e align %.2e, lengths %s" %
              ((name, B, T_enc) + tuple(errs) + (ref[4].tolist(),)))
        assert max(errs) < TOL, (name, errs)
        if impl == _capi.IMPL_PERSISTENT:
            # the energies of all rounds are summed in a fixed order: a second run is bit-identical
            memory = model.encoder.inference(sd["embedding.weight"][text].transpose(1, 2).cuda())
            runs = []
            for _ in range(2):
                with torch.no_grad(), t2.dropout_masks(prenet=keep):
                    runs.append([x.clone() for x in model.decoder.inference(memory)])
            assert all(torch.equal(a, b) for a, b in zip(*runs)), "persistent decoder is not bit-reproducible"
    if T_enc > STEPWISE_MAX_T_ENC:
        model = make_model(sd, steps, _capi.IMPL_STEPWISE)
        with torch.no_grad(), t2.dropout_masks(prenet=keep), pytest.raises(RuntimeError, match=STEPWISE_TOO_LONG):
            model.inference(text.cuda())
    print("   gate margin %.2e, %.1f s" % (margin, time.time() - t0))


def test_inference_beyond_the_persistent_limit_is_refused_cleanly():
    """T_enc = PERSISTENT_MAX_T_ENC + 1: IMPL_PERSISTENT refuses the shape; AUTO falls back to the stepwise kernel, which
    runs it if it fits there and otherwise refuses it too.  An error raises, returns no output and leaves the device
    usable."""
    T = PERSISTENT_MAX_T_ENC + 1
    sd = synth_state_dict(300, gate_bias=-10.0, scale=2.0)
    g = torch.Generator().manual_seed(4)
    memory = torch.randn(2, T, 512, generator=g)
    keep = keep_mask((3, 2, 2, 256), 0.5, 5)
    model = make_model(sd, 3)
    dec = model.decoder
    dec.mel_lengths = None
    eng = model._t2_engine()
    eng.impl = _capi.IMPL_PERSISTENT
    with torch.no_grad(), t2.dropout_masks(prenet=keep), pytest.raises(RuntimeError, match=PERSISTENT_REFUSED):
        dec.inference(memory.cuda())
    eng.impl = _capi.IMPL_AUTO
    with torch.no_grad(), t2.dropout_masks(prenet=keep):
        if T <= STEPWISE_MAX_T_ENC:
            out = dec.inference(memory.cuda())
            ref = O.decoder_inference(sd, memory, keep, 0.5, 3)
            assert rel_err(out[0], ref[0]) < TOL and rel_err(out[2], ref[2]) < TOL
        else:
            with pytest.raises(RuntimeError, match=STEPWISE_TOO_LONG):
                dec.inference(memory.cuda())
            assert dec.mel_lengths is None
    torch.cuda.synchronize()
    # the device and the model still work at the limit
    short = memory[:, :PERSISTENT_MAX_T_ENC].contiguous()
    with torch.no_grad(), t2.dropout_masks(prenet=keep):
        out = dec.inference(short.cuda())
        ref = O.decoder_inference(sd, short, keep, 0.5, 3)
    assert rel_err(out[0], ref[0]) < TOL and rel_err(out[2], ref[2]) < TOL


# ---- 2. / 3. teacher-forced forward + decoder backward ----------------------------------------------------------------
def engine_decoder_grads(model, case, training, gemm, monkeypatch):
    """gemm = tc: the reverse recurrence's GEMMs and the LSTM weight gradients on the tcgen05 engines (default); simt: the
    fp32 SIMT kernels and plain cuBLAS fp32 GEMMs."""
    monkeypatch.setenv("T2_BWD_GEMM", gemm)
    monkeypatch.setenv("T2_WGRAD", "tc" if gemm == "tc" else "cublas")
    memory, mels, lens, pk, ak, dk, d_mel, d_gate, d_align = case
    dec = model.train(training).decoder
    for p in dec.parameters():
        p.grad = None
    mem = memory.cuda().requires_grad_(True)
    with t2.dropout_masks(prenet=pk, att=ak, dec=dk):
        mel, gate, align = dec(mem, mels.cuda(), lens.cuda())
        loss = (mel * d_mel.cuda()).sum() + (gate * d_gate.cuda()).sum()
        if d_align is not None:
            loss = loss + (align * d_align.cuda()).sum()
        loss.backward()
    torch.cuda.synchronize()
    got = {"mel": mel, "gate": gate, "align": align, "d_memory": mem.grad}
    for k, p in dec.named_parameters():
        assert p.grad is not None, k
        got["decoder." + k] = p.grad
    return got


def oracle_decoder(sd, case, training, dtype):
    if dtype == torch.float64:
        sd = {k: (fp64(v) if k.startswith("decoder.") else v) for k, v in sd.items()}
        case = [fp64(x) for x in case]
    out, grads, dmem = oracle_decoder_grads(sd, *case, training)
    ref = {"mel": out[0], "gate": out[1], "align": out[2], "d_memory": dmem}
    ref.update(grads)
    return ref


def run_decoder_case(B, Te, T, training, use_align, lens, seed, monkeypatch, gemms=("tc",)):
    t0 = time.time()
    sd = synth_state_dict(seed=21, scale=2.0)
    case = list(decoder_case(B, Te, T, seed=seed))
    if lens is not None:
        case[2] = torch.tensor(lens, dtype=torch.long)
    if not use_align:
        case[8] = None
    r32 = oracle_decoder(sd, case, training, torch.float32)
    r64 = oracle_decoder(sd, case, training, torch.float64)
    t_oracle = time.time() - t0
    model = t2.Tacotron2(t2.create_hparams())
    model.load_state_dict(sd)
    model = model.cuda()
    res = {}
    for gemm in gemms:
        got = engine_decoder_grads(model, case, training, gemm, monkeypatch)
        check_vs_fp64("decoder backward [%s] B=%d T_enc=%d T_mel=%d" % (gemm, B, Te, T), got, r32, r64)
        # padded encoder positions get no gradient at all, exactly as in the oracle
        for b, n in enumerate(case[2].tolist()):
            if n < Te:
                assert float(r64["d_memory"][b, n:].abs().max()) == 0.0
                assert float(got["d_memory"][b, n:].abs().max()) == 0.0, (gemm, b, n)
        res[gemm] = {k: v.detach().clone() for k, v in got.items()}
    print("   oracle %.1f s, total %.1f s" % (t_oracle, time.time() - t0))
    return res


# (B, T_enc, T_mel, training, d_align, memory_lengths or None for ragged lengths in [T_enc / 2, T_enc])
BWD_CASES = [
    (2, 256, 7, False, True, None),                                  # 1 attention round
    (3, 257, 13, True, False, None),                                 # 2 rounds
    # row lengths in both rounds, on both sides of the 80 memory rows the forward stages in shared memory, and 1
    (7, 300, 9, False, False, (300, 257, 256, 81, 80, 17, 1)),
    (2, BWD_MAX_T_ENC, 11, True, True, None),
]


@pytest.mark.parametrize("B,Te,T,training,use_align,lens", BWD_CASES)
def test_decoder_backward_across_attention_rounds_vs_fp64_oracle(B, Te, T, training, use_align, lens, monkeypatch):
    run_decoder_case(B, Te, T, training, use_align, lens, 500 + Te, monkeypatch)


def test_decoder_backward_full_batch_at_the_limit_tc_vs_simt(monkeypatch):
    """B = 64 at T_enc = BWD_MAX_T_ENC, training mode, ragged lengths: both GEMM engines against the fp64 oracle and
    within 1e-4 of each other (as at T_enc = 150 in test_gpu_backward.py)."""
    res = run_decoder_case(64, BWD_MAX_T_ENC, 6, True, False, None, 64, monkeypatch, gemms=("tc", "simt"))
    worst = max(rel_err(res["tc"][k], res["simt"][k]) for k in res["tc"])
    print("   tcgen05 vs SIMT GEMMs worst rel diff %.2e" % worst)
    assert worst < 1e-4


# T_mel -> K splits of the LSTM weight gradients (wgrad_seg): 100 = one full split; 101 = a full split and a 1-step one;
# 250 = two full splits and a partial one; 1500 = 15 full splits; 1501 = the split widened to 150 steps: 11 splits, the
# last of 1 step, chains of 150 x 4 x 3 = 1800 MMAs
@pytest.mark.parametrize("B,T", [(2, 100), (2, 101), (2, 250), (1, 1500), (1, 1501)])
def test_decoder_weight_gradient_k_splits_vs_fp64_oracle(B, T, monkeypatch):
    run_decoder_case(B, 20, T, True, True, None, 700 + T, monkeypatch)


# ---- 4. whole training step at long text ------------------------------------------------------------------------------
def test_train_step_at_the_backward_t_enc_limit_vs_fp64_oracle():
    """Tacotron2.forward + Tacotron2Loss + backward at T_text = BWD_MAX_T_ENC (text lengths 408 and 230, T_mel = 160):
    the training-mode encoder convolutions and BatchNorm, the packed BiLSTM backward over 408 steps, the embedding gradient
    of long rows, the decoder backward at its T_enc limit.  Every parameter gradient and the loss."""
    t0 = time.time()
    B, Tt, Tm = 2, BWD_MAX_T_ENC, 160
    sd = synth_state_dict(seed=43, scale=2.0)
    text = rand_text(B, Tt, 8)
    tl = torch.tensor([Tt, 230])
    ol = torch.tensor([Tm, 117])
    g = torch.Generator().manual_seed(9)
    mels = torch.randn(B, 80, Tm, generator=g)
    gt = torch.zeros(B, Tm)
    for i, n in enumerate(ol.tolist()):
        mels[i, :, n:] = 0
        gt[i, n - 1:] = 1
    m = dict(pk=keep_mask((Tm + 1, 2, B, 256), 0.5, 1), ak=keep_mask((Tm, B, 1024), 0.1, 2), dk=keep_mask((Tm, B, 1024), 0.1, 3),
             ek=keep_mask((3, B, 512, Tt), 0.5, 4), qk4=keep_mask((4, B, 512, Tm), 0.5, 5), qk1=keep_mask((B, 80, Tm), 0.5, 6))
    loss32, _, g32 = oracle_train_step(sd, text, tl, ol, mels, gt, m, True)
    loss64, _, g64 = oracle_train_step(sd, text, tl, ol, mels, gt, m, True, dtype=torch.float64)
    t_oracle = time.time() - t0
    model = t2.Tacotron2(t2.create_hparams())
    model.load_state_dict(sd)
    model = model.cuda().train()
    post_keep = [m["qk4"][i] for i in range(4)] + [m["qk1"]]
    with t2.dropout_masks(prenet=m["pk"], att=m["ak"], dec=m["dk"], enc=m["ek"], post=post_keep):
        out = model((text.cuda(), tl.cuda(), mels.cuda(), Tt, ol.cuda()))
        loss = t2.Tacotron2Loss()(out, (mels.cuda(), gt.cuda()))
        loss.backward()
    torch.cuda.synchronize()
    loss_yard = abs(float(loss32) - float(loss64)) / abs(float(loss64))
    loss_err = abs(loss.item() - float(loss64)) / abs(float(loss64))
    print("train step B=%d T_text=%d T_mel=%d: loss %.6f, rel err %.2e (fp32 oracle %.2e)" %
          (B, Tt, Tm, loss.item(), loss_err, loss_yard))
    assert loss_err < max(1e-4, SLACK * loss_yard)
    got, r32, r64 = {}, {}, {}
    for k, p in model.named_parameters():
        assert p.grad is not None, k
        if k.endswith("0.conv.bias"):
            # a bias in front of a training-mode BatchNorm has an exactly-zero gradient; both sides hold rounding noise
            scale = float(g64[k.replace("0.conv.bias", "1.bias")].abs().max())
            assert float(p.grad.abs().max()) < 1e-3 * scale, k
            continue
        got[k], r32[k], r64[k] = p.grad, g32[k], g64[k]
    check_vs_fp64("train step B=%d T_text=%d T_mel=%d" % (B, Tt, Tm), got, r32, r64)
    print("   oracle %.1f s, total %.1f s" % (t_oracle, time.time() - t0))


# ---- 5. the backward's T_enc limit under autograd ---------------------------------------------------------------------
def test_decoder_beyond_the_backward_limit_under_autograd():
    """T_enc = BWD_MAX_T_ENC + 1: without autograd the teacher-forced forward still runs (and is right); under autograd the
    decoder and the whole model raise the library's "too long for the attention kernel" error no later than backward(), and
    no parameter is left with a partially written .grad."""
    Te, T, B = BWD_MAX_T_ENC + 1, 5, 2
    sd = synth_state_dict(seed=21, scale=2.0)
    memory, mels, lens, pk, ak, dk, _, _, _ = decoder_case(B, Te, T, seed=9)
    model = t2.Tacotron2(t2.create_hparams())
    model.load_state_dict(sd)
    model = model.cuda().train()
    dec = model.decoder
    with torch.no_grad(), t2.dropout_masks(prenet=pk, att=ak, dec=dk):
        out = dec(memory.cuda(), mels.cuda(), lens.cuda())
        ref = O.decoder_forward(sd, memory, mels, lens, pk.float(), ak.float(), dk.float(), training=True)
    for a, b in zip(out, ref):
        assert rel_err(a, b) < TOL
    with t2.dropout_masks(prenet=pk, att=ak, dec=dk), pytest.raises(RuntimeError, match=BWD_TOO_LONG):
        mem = memory.cuda().requires_grad_(True)
        mel, gate, _ = dec(mem, mels.cuda(), lens.cuda())
        (mel.sum() + gate.sum()).backward()
    assert mem.grad is None
    # the whole model: the postnet's backward runs before the decoder's, so the refusal has to come before either
    text = rand_text(B, Te, 3)
    tl = torch.tensor([Te, 300])
    ol = torch.tensor([T, T - 1])
    gt = torch.zeros(B, T)
    gt[0, -1] = 1
    gt[1, -2:] = 1
    with pytest.raises(RuntimeError, match=BWD_TOO_LONG):
        o = model((text.cuda(), tl.cuda(), mels.cuda(), Te, ol.cuda()))
        t2.Tacotron2Loss()(o, (mels.cuda(), gt.cuda())).backward()
    torch.cuda.synchronize()
    leaked = [k for k, p in model.named_parameters() if p.grad is not None]
    assert not leaked, leaked
