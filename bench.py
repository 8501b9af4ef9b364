#!/usr/bin/env python
"""bench.py -- mel frames/sec of the Tacotron 2 hot path (BASELINE.json configs[1]).

One "step" = one pass of the hot path over one batch: Tacotron2.inference on (B=64 per GPU,
T_text=150) synthetic text, exactly 800 decoder frames per row (gate_threshold = 1.0 so the stop
gate never fires, max_decoder_steps = 800; SURVEY.md section 8(d)) -> encoder, 800-step persistent
decoder, postnet.  51,200 mel frames per GPU per step.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

  value : frames/s with the text ids already resident in HBM (device tensors through the nn.Module API)
  e2e   : frames/s through the C-ABI t2_infer_host with HOST buffers (pinned text in, mel_postnet out)
  roofline     : the persistent decoder kernel, algorithmic FLOPs (38,350,592 per frame) / CUDA-event time
  cpu_baseline : the oracle port (oracle/tacotron2_oracle.py, torch CPU, all host threads) on a bounded sample
  --impl reference : the same metric from the CPU oracle port alone (the reference is pure Python; DESIGN.md
                     "reference arm")
  --dump-outputs DIR : after the timed steps, what the last timed Tacotron2.inference returned (rank 0's batch) as
                       DIR/<name>.npy, 63.7 MB in all; text, weights and dropout seeds are fixed, so two builds run with
                       the same arguments can be compared output for output
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_PER_GPU, T_TEXT, T_MEL = 64, 150, 800
FLOP_PER_FRAME = 2 * (18167296 + 6720 * T_TEXT)          # SURVEY.md section 8(d): 38,350,592 @ T_enc=150
STREAM_BYTES_PER_STEP = 97.3e6                           # fp32 weights + memory + processed memory
WORKLOAD = ("Tacotron2.inference: B=64 per GPU, T_text=150, 800 decoder frames per row (gate_threshold=1.0, "
            "max_decoder_steps=800), encoder + decoder + postnet; BASELINE.json configs[1]")


def synth_weights(seed=1234):
    from tests.common import synth_state_dict
    return synth_state_dict(seed, gate_bias=0.0, scale=1.0)


def load_max_mhz():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["sm_max_mhz"])
    except Exception:
        return 1965.0


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 6:
                    self.rows.append(parts)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None, "reasons": reasons,
                "samples": len(self.rows)}


def host_threads():
    """Threads this process may actually run on (the affinity mask, not the machine's core count)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def _best_threads(fn, candidates):
    """Runs fn() under each thread count and returns (best_seconds, best_threads)."""
    best = None
    for th in candidates:
        torch.set_num_threads(th)
        fn()                                  # warm-up at this thread count
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, th)
    return best


class CpuPort:
    """The oracle port (the reference's algorithm in plain torch CPU ops, oracle/tacotron2_oracle.py) on the host
    cores, on the SAME workload as the GPU arm: encoder + 800 decoder steps + postnet at B=64, T_text=150.  The thread
    count of each component (<= the affinity mask; small recurrent GEMMs are slower with 100+ threads than with 16) is
    tuned ONCE on small slices; a pass then either runs all 800 decoder steps or, when `dec_steps` < 800, that many
    steps extrapolated linearly (every step does identical work) -- the sample size is stated in the result."""

    def __init__(self):
        from oracle import tacotron2_oracle as O
        from tests.common import keep_mask, rand_text
        self.O = O
        self.threads = host_threads()
        cands = sorted({t for t in (8, 16, 32, 64, self.threads) if t <= self.threads})
        self.sd = synth_weights()
        text = rand_text(B_PER_GPU, T_TEXT, 1)
        self.keep = keep_mask((T_MEL, 2, B_PER_GPU, 256), 0.5, 2)
        self.mel = torch.randn(B_PER_GPU, 80, T_MEL)
        with torch.no_grad():
            self.emb = self.sd["embedding.weight"][text].transpose(1, 2)
            _, self.th_enc = _best_threads(lambda: O.encoder(self.sd, self.emb[:, :, :30]), cands)
            torch.set_num_threads(self.th_enc)
            self.memory = O.encoder(self.sd, self.emb)
            self.st0 = O.init_decoder_state(self.sd, self.memory)
            _, self.th_dec = _best_threads(lambda: self._steps(6), cands)
            _, self.th_post = _best_threads(lambda: O.postnet(self.sd, self.mel[:, :, :100]), cands)

    def _steps(self, n):
        O, sd = self.O, self.sd
        st = {k: v.clone() for k, v in self.st0.items()}
        x = self.memory.new_zeros(B_PER_GPU, 80)
        ts = []
        for t in range(n):
            t0 = time.perf_counter()
            px = O.prenet(sd, x, self.keep[t, 0], self.keep[t, 1])
            x, _, _ = O.decode_step(sd, st, self.memory, px)
            ts.append(time.perf_counter() - t0)
        return ts

    def run(self, dec_steps=T_MEL):
        """One pass; returns (cpu_baseline dict, seconds for the whole 51,200-frame workload)."""
        O, sd = self.O, self.sd
        dec_steps = min(int(dec_steps), T_MEL)
        with torch.no_grad():
            torch.set_num_threads(self.th_enc)
            t0 = time.perf_counter()
            O.encoder(sd, self.emb)
            t_enc = time.perf_counter() - t0
            torch.set_num_threads(self.th_dec)
            ts = self._steps(dec_steps)
            if dec_steps == T_MEL:
                t_dec, how = sum(ts), "all 800 decoder steps measured"
            else:
                body = sorted(ts[min(3, dec_steps // 4):])
                t_dec = T_MEL * body[len(body) // 2]
                how = "median of %d decoder steps x 800 (extrapolated)" % dec_steps
            torch.set_num_threads(self.th_post)
            t0 = time.perf_counter()
            O.postnet(sd, self.mel)
            t_post = time.perf_counter() - t0
        total = t_enc + t_dec + t_post
        return {"value": B_PER_GPU * T_MEL / total, "unit": "mel frames/s", "cores": max(self.th_enc, self.th_dec, self.th_post),
                "kind": "port",
                "sample": "oracle port, B=64 T_text=150, fp32, %d host threads usable: encoder %.3f s (%d thr) + decoder %.3f s "
                          "(%s, %d thr) + postnet T_mel=800 %.3f s (%d thr)"
                          % (self.threads, t_enc, self.th_enc, t_dec, how, self.th_dec, t_post, self.th_post),
                "decoder_step_us": t_dec / T_MEL * 1e6, "decoder_steps_measured": dec_steps}, total


def run_reference(args, rank):
    """--impl reference: the reference's algorithm on the host cores (the oracle port: the reference is pure Python and
    /root/reference does not exist on the GPU box), same metric / config as the GPU arm.  The first warm-up pass runs the
    complete workload; if K such passes would not fit ~4 minutes the timed passes measure a bounded number of decoder steps
    and extrapolate (stated in config.workload)."""
    if rank != 0:
        return
    t_start = time.perf_counter()
    port = CpuPort()
    cb, full_s = port.run(T_MEL)                      # warm-up pass 1: the whole workload, nothing extrapolated
    for _ in range(max(args.warmup - 1, 0)):
        port.run(40)
    budget = 240.0 - (time.perf_counter() - t_start)
    dec_steps = T_MEL if full_s * args.steps <= budget else max(40, int(T_MEL * budget / (full_s * args.steps)) // 10 * 10)
    vals = [port.run(dec_steps) for _ in range(args.steps)]
    vals.sort(key=lambda v: v[1])
    cb = vals[len(vals) // 2][0]
    ms = sum(v[1] for v in vals) / len(vals) * 1e3
    cb["full_pass_s"] = full_s
    line = {"impl": "reference", "metric": "mel frames/sec (B=64,T_text=150)", "value": cb["value"], "unit": "mel frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            # same workload string as the GPU arm (the driver compares the two configs); how this arm ran it is in `arm`
            "config": {"workload": WORKLOAD, "global_batch": B_PER_GPU * max(args.gpus, 1),
                       "arm": "oracle port on the host CPU cores (one host works through the %d shard(s) of 64 rows one after the "
                              "other: its frames/s does not depend on N), %s per timed pass"
                              % (max(args.gpus, 1), "all 800 decoder steps" if dec_steps == T_MEL else
                                 "%d of 800 decoder steps measured, extrapolated linearly" % dec_steps)},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "mel frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t_start}
    print(json.dumps(line))


def decoder_traffic():
    """DRAM bytes per decoder step of the persistent kernel from the committed ncu capture (profiles/decoder_traffic.json,
    written by tools/ncu_summary.py) -- valid only for the kernel source it was captured from: a stale hash gives None."""
    import hashlib
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "decoder_traffic.json")))
        src = open(os.path.join(ROOT, "tacotron2_b200", "csrc", "decoder_persistent.cu"), "rb").read()
        if hashlib.sha256(src).hexdigest()[:16] != d.get("source_sha16"):
            return None, "profiles/decoder_traffic.json is stale (kernel source changed since the capture)"
        return float(d["dram_bytes_per_step"]), d.get("capture")
    except Exception as e:
        return None, "unavailable: %s" % str(e)[:80]


def train_inputs(B, Tt, Tm, seed):
    """SURVEY.md section 8(d) config 3: sorted text lengths U[Tt/2, Tt] (max = Tt), mel ~ N(0,1), output lengths
    U[Tm/2, Tm] (max = Tm), zero-padded targets, gate target 1 from the last frame on (data_utils.py:97-107)."""
    g = torch.Generator().manual_seed(seed)
    text = torch.randint(0, 148, (B, Tt), generator=g)
    tl = torch.sort(torch.randint(Tt // 2, Tt + 1, (B,), generator=g), descending=True)[0]
    tl[0] = Tt
    ol = torch.randint(Tm // 2, Tm + 1, (B,), generator=g)
    ol[0] = Tm
    mels = torch.randn(B, 80, Tm, generator=g)
    gt = torch.zeros(B, Tm)
    for i, n in enumerate(ol.tolist()):
        mels[i, :, n:] = 0
        gt[i, n - 1:] = 1
    return text, tl, mels, gt, ol


def train_block(t2, hp, rank, world, iters=3, warmup=2):
    """BASELINE.json configs[2] / configs[3], measured AFTER the headline region: one teacher-forced training step
    (Tacotron2.forward + Tacotron2Loss + backward + clip + Adam, train.py:209-236) at B=64 per GPU, T_text=150,
    T_mel=800; with N > 1 the same step under apply_gradient_allreduce (bucketed NCCL all-reduce launched from the
    backward hooks, distributed.py:126-173).  Times are CUDA events, max over ranks.  exposed all-reduce = DP step -
    local step on the same ranks."""
    import torch.distributed as dist
    from tacotron2_b200.distributed import apply_gradient_allreduce
    torch.manual_seed(1234)
    model = t2.Tacotron2(hp)
    model.load_state_dict(synth_weights())
    model = model.cuda().train()
    opt = t2.FusedClipAdam(model.parameters(), lr=hp.learning_rate, weight_decay=hp.weight_decay)
    crit = t2.Tacotron2Loss()
    text, tl, mels, gt, ol = (x.cuda() for x in train_inputs(B_PER_GPU, T_TEXT, T_MEL, 1234 + rank))
    x = (text, tl, mels, int(tl.max()), ol)

    def one_step():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        model.zero_grad(set_to_none=True)
        out = model(x)
        loss = crit(out, (mels, gt))
        ev[1].record()
        loss.backward()
        ev[2].record()
        opt.step(max_norm=hp.grad_clip_thresh)
        ev[3].record()
        ev[3].synchronize()
        return [ev[i].elapsed_time(ev[i + 1]) for i in range(3)], float(loss)

    def timed_steps():
        for _ in range(warmup):
            one_step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        rows = [one_step() for _ in range(iters)]
        rows.sort(key=lambda r: sum(r[0]))
        med = rows[len(rows) // 2]                                                 # the median step (by total time)
        t = torch.tensor(med[0], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.cpu()], rows[-1][1]

    L = _launch_counter()
    l0 = L()
    local, loss = timed_steps()
    launches = (L() - l0) // (iters + warmup)
    n_param = sum(p.numel() for p in model.parameters())
    out = {"workload": "teacher-forced training step B=64 per GPU, T_text=150, T_mel=800, fp32-grade (split-fp16 tensor-core "
                       "operands), fwd + loss + bwd + clip + Adam; BASELINE.json configs[2]",
           "ms_per_step": sum(local), "forward_loss_ms": local[0], "backward_ms": local[1], "clip_adam_ms": local[2],
           "frames_per_s": B_PER_GPU * T_MEL * world / (sum(local) * 1e-3) if world == 1 else None,
           "loss": loss, "gpu_launches_per_step": int(launches), "max_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}
    if world > 1:
        apply_gradient_allreduce(model)
        dp, _ = timed_steps()
        out.update({"workload": out["workload"].replace("configs[2]", "configs[3]: data parallel, NCCL gradient all-reduce"),
                    "local_ms_per_step": sum(local), "ms_per_step": sum(dp), "forward_loss_ms": dp[0], "backward_ms": dp[1],
                    "clip_adam_ms": dp[2], "allreduce_exposed_ms": sum(dp) - sum(local),
                    "allreduce_bytes": n_param * 4, "frames_per_s": B_PER_GPU * T_MEL * world / (sum(dp) * 1e-3),
                    "dp_efficiency_vs_local_step": sum(local) / sum(dp)})
    del model, opt
    torch.cuda.empty_cache()
    return out


def config5_block(t2, hp, rank, world, iters=3):
    """BASELINE.json configs[4]: long-sequence inference B=256 over 8 GPUs = 32 rows per GPU, T_text=300, 2000 decoder
    steps (gate_threshold = 1.0); per-GPU share measured on every rank, max over ranks."""
    import contextlib
    import torch.distributed as dist
    from tests.common import rand_text
    model = t2.Tacotron2(hp)
    model.load_state_dict(synth_weights())
    model = model.cuda().eval()
    model.decoder.max_decoder_steps, model.decoder.gate_threshold = 2000, 1.0
    text = rand_text(32, 300, 200 + rank).cuda()
    ms = []
    for it in range(iters + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        with torch.no_grad(), contextlib.redirect_stdout(sys.stderr):
            out = model.inference(text)
        e1.record()
        e1.synchronize()
        if it:
            ms.append(e0.elapsed_time(e1))
    assert out[0].shape == (32, 80, 2000)
    ms.sort()
    t = torch.tensor([ms[len(ms) // 2]], device="cuda", dtype=torch.float64)      # median of the timed iterations
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    m = float(t.cpu())
    del model
    torch.cuda.empty_cache()
    return {"workload": "Tacotron2.inference B=32 per GPU, T_text=300, 2000 decoder frames per row; BASELINE.json configs[4] "
                        "(B=256 over 8 GPUs)", "ms_per_batch": m, "frames_per_s": 32 * 2000 * world / (m * 1e-3),
            "decoder_step_us": None}


def eager_gpu_context():
    """Context only (SURVEY.md 8(d)): the oracle port -- plain torch ops, what stock PyTorch eager does with this model --
    on cuda:0, outside every timed region of the GPU arm: encoder + 60 decoder steps (extrapolated to 800) + postnet."""
    try:
        from oracle import tacotron2_oracle as O
        from tests.common import keep_mask, rand_text
        sd = {k: v.cuda() for k, v in synth_weights().items()}
        text = rand_text(B_PER_GPU, T_TEXT, 1).cuda()
        keep = keep_mask((64, 2, B_PER_GPU, 256), 0.5, 2).cuda()
        with torch.no_grad():
            emb = sd["embedding.weight"][text].transpose(1, 2)
            memory = O.encoder(sd, emb)
            mel = torch.randn(B_PER_GPU, 80, T_MEL, device="cuda")
            res = {}
            for rep in range(2):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                memory = O.encoder(sd, emb)
                torch.cuda.synchronize()
                t_enc = time.perf_counter() - t0
                st = O.init_decoder_state(sd, memory)
                x = memory.new_zeros(B_PER_GPU, 80)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for t in range(60):
                    px = O.prenet(sd, x, keep[t, 0], keep[t, 1])
                    x, _, _ = O.decode_step(sd, st, memory, px)
                torch.cuda.synchronize()
                t_step = (time.perf_counter() - t0) / 60
                t0 = time.perf_counter()
                O.postnet(sd, mel)
                torch.cuda.synchronize()
                t_post = time.perf_counter() - t0
                res = {"frames_per_s": B_PER_GPU * T_MEL / (t_enc + T_MEL * t_step + t_post), "decoder_step_us": t_step * 1e6,
                       "encoder_ms": t_enc * 1e3, "postnet_ms": t_post * 1e3,
                       "what": "oracle port (plain torch fp32 ops, TF32 off) on cuda:0, 60 decoder steps extrapolated to 800; context only"}
        return res
    except Exception as e:
        return {"unavailable": str(e)[:120]}


def dump_outputs(out_dir, arrays):
    """Writes name -> tensor as out_dir/<name>.npy: floating-point tensors as float32, integer ones as float64."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().cpu()
        np.save(os.path.join(out_dir, name + ".npy"), (t.float() if t.is_floating_point() else t.double()).numpy())


def _launch_counter():
    from tacotron2_b200 import _capi
    return _capi.lib().t2_kernel_launch_count


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--decoder-impl", default="auto", choices=["auto", "stepwise", "persistent"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the train / config5 / eager_gpu blocks (A/B runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the GPU path; the reference arm has none")
        run_reference(args, rank)
        return
    args.warmup = max(args.warmup, 3)
    # the engine's Philox dropout seeds derive from torch.initial_seed(), which is random per process unless set: fixed,
    # runs with the same arguments compute the same outputs
    torch.manual_seed(1234)

    import torch.distributed as dist
    import tacotron2_b200 as t2
    from tacotron2_b200 import _capi
    from tests.common import rand_text
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    hp = t2.create_hparams()
    model = t2.Tacotron2(hp)
    model.load_state_dict(synth_weights())
    model = model.cuda().eval()
    model.decoder.max_decoder_steps = T_MEL
    model.decoder.gate_threshold = 1.0            # sigmoid(.) > 1.0 never fires -> exactly 800 frames per row
    eng = model._t2_engine()
    eng.impl = {"auto": _capi.IMPL_AUTO, "stepwise": _capi.IMPL_STEPWISE, "persistent": _capi.IMPL_PERSISTENT}[args.decoder_impl]
    L = _capi.lib()

    text = rand_text(B_PER_GPU, T_TEXT, 100 + rank)
    text_dev = text.cuda()
    text_host = text.clone().pin_memory()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")    # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, iters):
        """Per-iteration CUDA-event timing (L2 flushed, untimed, between iterations)."""
        total = 0.0
        for _ in range(iters):
            flush.fill_(1)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            total += e0.elapsed_time(e1)
        return total

    import contextlib

    last_out = None

    def step_device():
        nonlocal last_out
        # the reference prints "Warning! Reached max decoder steps" to stdout (model.py:446); this
        # workload reaches the cap by construction, keep stdout for the single JSON line
        with torch.no_grad(), contextlib.redirect_stdout(sys.stderr):
            last_out = model.inference(text_dev)

    out_host = None

    def step_host():
        nonlocal out_host
        out_host = eng.infer_host(text_host, T_MEL, 1.0, out_host=out_host)

    # component timers (rank-local, for the roofline / breakdown)
    def decoder_only():
        with torch.no_grad():
            return eng.decoder(memory_dev, _capi.MODE_INFER, T_MEL, gate_threshold=1.0)

    with torch.no_grad():
        memory_dev = eng.encoder(text=text_dev)
    for _ in range(args.warmup):
        step_device(); step_host()
    barrier()
    sampler = ClockSampler(local_rank); sampler.start()
    launches0 = L.t2_kernel_launch_count()
    ms_dev = timed(step_device, args.steps)
    launches = L.t2_kernel_launch_count() - launches0
    if args.dump_outputs and rank == 0:      # before any other call can reuse the engine's buffers
        dump_outputs(args.dump_outputs, dict(zip(("mel_outputs", "mel_outputs_postnet", "gate_outputs", "alignments"), last_out),
                                             mel_lengths=model.mel_lengths))
    last_out = None
    barrier()
    ms_e2e = timed(step_host, args.steps)
    barrier()
    ms_dec = timed(decoder_only, args.steps)
    sampler.stop_flag = True
    phase_profile = None
    try:
        prof = eng.decoder_profile()
        tot = sum(v[0] for v in prof.values()) or 1
        sm_mhz = float((sampler.summary().get("sm_mhz") or 0) or load_max_mhz())     # clock64 ticks at the SM clock
        phase_profile = {k: {"us_per_step_cta0_60_100": [round(x / sm_mhz / T_MEL, 2) for x in v]} for k, v in prof.items()}
        phase_profile["sm_mhz_used"] = sm_mhz
    except Exception as e:  # stepwise implementation has no phase profile
        phase_profile = {"unavailable": str(e)[:80]}
    n_frames = int(out_host[2][0]) * B_PER_GPU
    assert n_frames == B_PER_GPU * T_MEL, "workload did not produce 800 frames per row: %d" % n_frames
    extras = None
    if not args.no_extras:       # after (and outside) the headline region; every rank takes part (DP all-reduce at N > 1)
        del flush
        torch.cuda.empty_cache()
        extras = {"train": train_block(t2, hp, rank, world), "config5": config5_block(t2, hp, rank, world)}
    t = torch.tensor([ms_dev, ms_e2e, ms_dec], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e, ms_dec = (float(x) for x in t.cpu())
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    frames = B_PER_GPU * T_MEL * world * args.steps
    value = frames / (ms_dev * 1e-3)
    e2e = frames / (ms_e2e * 1e-3)
    peak_tf, peak_gbs, peak_src = load_peaks()
    traffic_step, traffic_src = decoder_traffic()
    dec_s = ms_dec * 1e-3 / args.steps
    ach_tf = B_PER_GPU * T_MEL * FLOP_PER_FRAME / dec_s / 1e12
    ach_gbs = T_MEL * STREAM_BYTES_PER_STEP / dec_s / 1e9
    info = (torch.cuda.get_device_name(0))
    line = {
        "metric": "mel frames/sec (B=64,T_text=150)", "value": value, "unit": "mel frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (split-fp16 tensor-core operands hi+lo, fp32 accumulate and state)", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "global_batch": B_PER_GPU * world, "parallelism": "dp%d (batch sharded, no collective)" % world,
                   "l2": "256 MiB flush between timed iterations", "decoder_impl": args.decoder_impl, "device": info},
        "e2e": {"value": e2e, "unit": "mel frames/s", "h2d_bytes_per_step": B_PER_GPU * T_TEXT * 8,
                "d2h_bytes_per_step": B_PER_GPU * 80 * T_MEL * 4 + B_PER_GPU * 4 + 4, "ms_per_step": ms_e2e / args.steps,
                "returns": "mel_outputs_postnet (B,80,800) fp32 + mel_lengths (B) + n_steps -- what the vocoder consumes; "
                           "the reference's inference() also returns mel_outputs, gate and alignments (+51 MB), which stay on "
                           "the device here"},
        "gpu_launches": int(launches),
        "decoder_step_us": dec_s / T_MEL * 1e6, "decoder_ms": dec_s * 1e3,
        "roofline": {"bound": "tensor", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf,
                     # dram__bytes_read + write of the persistent kernel per launch, from the committed ncu --set full capture of
                     # THIS kernel source (profiles/decoder_traffic.json; null when the source changed since)
                     "traffic": traffic_step * T_MEL if traffic_step else None, "traffic_source": traffic_src, "kernel": "decoder (persistent kernel + processed_memory GEMM), CUDA events",
                     "peak_source": peak_src, "algorithmic_flop_per_frame": FLOP_PER_FRAME,
                     "stream_bytes": {"achieved_GBps": ach_gbs, "peak_GBps": peak_gbs, "frac": ach_gbs / peak_gbs,
                                      "bytes_per_step": STREAM_BYTES_PER_STEP}},
        "clocks": sampler.summary(),
        "decoder_phase_profile": phase_profile,
    }
    if extras is not None:
        line.update(extras)
    if not args.no_cpu_baseline and world == 1:
        port = CpuPort()
        port.run(20)                                     # warm-up
        cb, _ = port.run(100)                            # bounded sample: ~10-30 s of CPU work including the tuning
        line["cpu_baseline"] = cb
        line["eager_gpu"] = eager_gpu_context()
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
