#!/usr/bin/env python
"""Benchmark of the hot path: utterances/sec of one training step (zero_grad -> forward -> label-smoothed CE ->
backward -> single gradient all-reduce -> Adam) of the speech Transformer, BASELINE.json cfg2 per GPU:
4 layers / 8 heads / d=512 / d_ff=2048 / vgg_cnn, batch 32, T_src=800 x 161 mel, T_tgt=100, V=4364, dropout 0.1.

    python bench.py --gpus N --steps K --warmup W                 # ours  (torchrun launches N>1)
    python bench.py --impl reference --gpus N --steps K --warmup W    # the reference algorithm on the host CPU
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # + the last timed step's outputs as DIR/*.npy

Prints ONE JSON line (see the task contract): `value` = whole-job utt/s with inputs resident in HBM, `e2e` = the same
step through the public API with pinned-host inputs copied in and the loss read back every step, `roofline` for the
dominant kernel group (CUDA-event timed on the launching stream inside the timed region), `cpu_baseline` = the oracle
port on the host cores (rank 0, N=1).  Data are synthetic, weights random-init (no network for corpora/checkpoints).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOAD = "cfg2"
METRIC = "utterances/sec (fwd+bwd) dim512/4L/8H T_src=800"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.proc, self.index, self.first = [], None, index, 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self):
        self.first = len(self.rows)

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        rows = self.rows[self.first:] or self.rows[-3:]     # a very short timed region can fall between two samples
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=(max(mx) if mx else None), reasons=sorted(reasons),
                    samples=len(sm))


# ---------------------------------------------------------------------------------------------------- algorithmic work
def algorithmic_flops(name, a):
    """FLOPs of one C-ABI call from its raw arguments (formulae of SURVEY.md §8d)."""
    if name == "linear_fwd" or name == "linear_bwd_data" or name == "linear_bwd_weight":
        M, N, K = a[4], a[5], a[6]
        return 2.0 * M * N * K
    if name == "conv3x3_fwd":
        B, T, F, Ci, Co = a[5], a[6], a[7], a[8], a[9]
        return 2.0 * 9 * B * T * F * Ci * Co
    if name == "conv3x3_fwd_pool":                               # x, w, bias, y, pooled, pool_idx, ws, then the dims
        B, T, F, Ci, Co = a[7], a[8], a[9], a[10], a[11]
        return 2.0 * 9 * B * T * F * Ci * Co
    if name in ("conv3x3_bwd_data", "conv3x3_bwd_weight"):       # one more pointer (the bf16 pair output / input) before the dims
        B, T, F, Ci, Co = a[6], a[7], a[8], a[9], a[10]
        return 2.0 * 9 * B * T * F * Ci * Co
    if name == "conv3x3_c1_fwd" or name == "conv3x3_c1_bwd_weight":
        off = 4
        B, F, T, Co = a[off], a[off + 1], a[off + 2], a[off + 3]
        return 2.0 * 9 * B * T * F * Co
    if name == "sdpa_fwd":
        B, H, Tq, Tk, dk, dv = a[20:26]
        return 2.0 * B * H * Tq * Tk * (dk + dv)
    if name == "sdpa_bwd":
        B, H, Tq, Tk, dk, dv = a[25:31]
        return 2.0 * 2.0 * B * H * Tq * Tk * (dk + dv)      # four GEMMs (recompute of QK^T not counted)
    if name == "sdpa_mat_fwd":      # q,k,v + 9 strides + key_pad, dense, causal, out + 3 strides, probs, probs_drop, then dims
        B, H, Tq, Tk, dk, dv = a[21:27]
        return 2.0 * B * H * Tq * Tk * (dk + dv)
    if name == "sdpa_fused_fwd":    # q,k,v + 9 strides + key_pad, dense, causal, out + 3 strides, lse, ws16, then dims
        B, H, Tq, Tk, dk, dv = a[21:27]
        return 2.0 * B * H * Tq * Tk * (dk + dv)
    if name == "sdpa_fused_bwd":    # dout,q,k,v,out,lse + 12 strides + key_pad, dense, causal + dq,dk,dv + ws16, ws_bwd, then dims
        B, H, Tq, Tk, dk, dv = a[26:32]
        return 2.0 * 2.0 * B * H * Tq * Tk * (dk + dv)
    if name == "sdpa_mat_bwd":      # dout,q,k,v + 12 strides + 6 pointers, then dims
        B, H, Tq, Tk, dk, dv = a[22:28]
        return 2.0 * 2.0 * B * H * Tq * Tk * (dk + dv)
    return 0.0


def summarize_profile(report, steps, peaks):
    groups = []
    for name, calls in report.items():
        ms = sum(t for _, t in calls) / steps
        fl = sum(algorithmic_flops(name, a) for a, _ in calls) / steps
        groups.append(dict(kernel=name, launches_per_step=len(calls) / steps, ms_per_step=ms, gflop_per_step=fl / 1e9))
    groups.sort(key=lambda g: -g["ms_per_step"])
    tot = sum(g["ms_per_step"] for g in groups)
    for g in groups:
        g["share"] = g["ms_per_step"] / tot if tot else 0.0
        g["tflops"] = g["gflop_per_step"] / g["ms_per_step"] if g["ms_per_step"] else 0.0
    return groups


# ---------------------------------------------------------------------------------------------------- CPU arm
def host_threads():
    """Threads for the CPU arm: the PHYSICAL cores this process may use (torch's own default; one thread per hardware
    thread -- 128 on the 64-core GPU box -- was measured 30x slower), also under torchrun, which exports OMP_NUM_THREADS=1,
    and never more than a cgroup CPU quota allows."""
    n = None
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
    except Exception:
        pass
    logical = len(os.sched_getaffinity(0))
    n = min(n or max(1, logical // 2), logical)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def cpu_oracle_throughput(batch, steps, warmup, threads=None):
    """Oracle port (oracle/asr_oracle.py: the reference's algorithm restated on torch CPU kernels) fwd+bwd utt/s."""
    from oracle import asr_oracle as O
    import b200asr
    torch.set_num_threads(threads or host_threads())
    c = b200asr.BASELINE_CONFIGS[WORKLOAD]["cfg"]
    ocfg = O.OracleConfig(num_layers=c.num_layers, num_heads=c.num_heads, dim_model=c.dim_model, dim_key=c.dim_key,
                          dim_value=c.dim_value, dim_inner=c.dim_inner, vocab=c.vocab, feat_extractor=c.feat_extractor,
                          tgt_max_len=c.tgt_max_len, freq=c.freq)
    P = O.init_params(ocfg, seed=123456)
    src, lens, tgt = O.synthetic_batch(ocfg, batch, b200asr.BASELINE_CONFIGS[WORKLOAD]["t_src"], seed=0, ragged=False)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.forward_backward(P, ocfg, src, lens, tgt, c.label_smoothing)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    mean = sum(times) / len(times)
    return batch / mean, mean, torch.get_num_threads()


def reference_flags(cfg, cuda=False):
    """The reference's own command-line flags (utils/constant.py) for an ASRConfig."""
    f = ["--num-layers", cfg.num_layers, "--num-heads", cfg.num_heads, "--dim-model", cfg.dim_model, "--dim-emb", cfg.dim_model,
         "--dim-key", cfg.dim_key, "--dim-value", cfg.dim_value, "--dim-inner", cfg.dim_inner, "--feat_extractor", cfg.feat_extractor,
         "--tgt-max-len", cfg.tgt_max_len, "--src-max-len", cfg.src_max_len, "--dropout", cfg.dropout,
         "--label-smoothing", cfg.label_smoothing, "--warmup", 4000, "--min-lr", 1e-6, "--k-lr", 1]
    return [str(x) for x in f] + (["--cuda"] if cuda else [])


def build_reference(cfg, cuda=False):
    """The UNMODIFIED reference model + its own optimizer (utils/functions.py:101-152), imported from /root/reference or the
    staged oracle/_ref (oracle/make_ref.py).  Returns (namespace, model, opt) or None when the checkout is absent."""
    from oracle import ref_shim
    if not ref_shim.available():
        return None
    ns = ref_shim.load(reference_flags(cfg, cuda))
    l2i, i2l = ref_shim.labels(cfg.vocab)
    torch.manual_seed(123456)
    model = ns.functions.init_transformer_model(ns.constant.args, l2i, i2l)
    if cuda:
        model = model.cuda()
    model.train()
    opt = ns.functions.init_optimizer(ns.constant.args, model, "noam")
    return ns, model, opt


def reference_step(ns, model, opt, src, lens, tgt, smoothing):
    """One iteration of the reference's training loop, trainer/asr/trainer.py:56-111 minus the string metrics:
    zero_grad -> model(...) -> calculate_metrics -> loss.backward() -> opt.step()."""
    opt.zero_grad()
    pred, gold, hyp, _ = model(src, lens, tgt, verbose=False)
    loss, _ = ns.metrics.calculate_metrics(pred, gold, smoothing=smoothing, loss_type="ce")
    loss.backward()
    opt.step()
    return loss


def cpu_reference_throughput(batch, steps, warmup, threads=None):
    """The reference's own PyTorch CPU path (kind "reference") on a `batch`-utterance sample of the workload; falls back to
    the oracle port (kind "port") only if the reference checkout is not staged."""
    import b200asr
    spec = b200asr.BASELINE_CONFIGS[WORKLOAD]
    cfg = spec["cfg"]
    torch.set_num_threads(threads or host_threads())
    built = build_reference(cfg, cuda=False)
    if built is None:
        ups, mean, thr = cpu_oracle_throughput(batch, steps, warmup, threads)
        return ups, mean, thr, "port"
    ns, model, opt = built
    g = torch.Generator().manual_seed(0)
    src = torch.randn(batch, 1, cfg.freq, spec["t_src"], generator=g)
    tgt = torch.randint(3, cfg.vocab, (batch, cfg.tgt_max_len - 1), generator=g)
    lens = torch.full((batch,), spec["t_src"], dtype=torch.int32)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        reference_step(ns, model, opt, src, lens, tgt, cfg.label_smoothing)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    mean = sum(times) / len(times)
    return batch / mean, mean, torch.get_num_threads(), "reference"


def gpu_reference_throughput(dev, batch, steps=5, warmup=3):
    """The unmodified reference, eager, ON THE SAME B200 (SURVEY.md 8d: "the kernel-for-kernel bar"): same step as
    reference_step, inputs resident on the device, CUDA-event timed; once with PyTorch's default flags (cuDNN convolutions
    may use TF32, matmuls are fp32) and once with allow_tf32 everywhere.  None when the checkout is not staged."""
    import b200asr
    spec = b200asr.BASELINE_CONFIGS[WORKLOAD]
    cfg = spec["cfg"]
    out = {}
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    try:
        for name, conv_tf32, mm_tf32 in (("fp32_strict", False, False), ("torch_default", True, False), ("allow_tf32", True, True)):
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = conv_tf32, mm_tf32
            built = build_reference(cfg, cuda=True)
            if built is None:
                return None
            ns, model, opt = built
            g = torch.Generator().manual_seed(0)
            src = torch.randn(batch, 1, cfg.freq, spec["t_src"], generator=g).to(dev)
            tgt = torch.randint(3, cfg.vocab, (batch, cfg.tgt_max_len - 1), generator=g).to(dev)
            lens = torch.full((batch,), spec["t_src"], dtype=torch.int32)
            for _ in range(warmup):
                reference_step(ns, model, opt, src, lens, tgt, cfg.label_smoothing)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                loss = reference_step(ns, model, opt, src, lens, tgt, cfg.label_smoothing)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[name] = {"ms_per_step": ms, "value": batch / (ms / 1e3), "unit": "utt/s", "cudnn_allow_tf32": conv_tf32,
                         "matmul_allow_tf32": mm_tf32, "loss": float(loss.item())}
            del model, opt, src, tgt
            torch.cuda.empty_cache()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
    out["note"] = (f"unmodified reference (oracle/_ref) eager on this GPU, batch {batch}, zero_grad+fwd+calculate_metrics+bwd+"
                   f"NoamOpt/Adam step, {steps} timed steps after {warmup} warm-up; torch {torch.__version__}")
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    b = 8            # bounded sample: a quarter of the cfg2 batch per step (~3 s of CPU work), enough rows to keep all cores busy
    ups, mean, threads, kind = cpu_reference_throughput(b, args.steps, args.warmup)
    what = "the unmodified reference (oracle/_ref)" if kind == "reference" else "oracle port"
    out = {"impl": "reference", "metric": METRIC, "value": ups, "unit": "utt/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": mean * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": WORKLOAD, "sample": f"{b} utterances per step of the cfg2 shape (T_src=800, T_tgt=100)",
                      "step": "zero_grad+fwd+CE+bwd+adam", "dropout": 0.1, "label_smoothing": 0.1},
           "cpu_baseline": {"value": ups, "unit": "utt/s", "cores": threads, "kind": kind,
                            "sample": f"{what}: training step on {b} utterances/step, {args.steps} steps"},
           "e2e": {"value": ups, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


# ---------------------------------------------------------------------------------------------------- GPU arm
DUMP_SAMPLE = 1 << 19        # elements of the parameter / gradient buffers written by --dump-outputs (fixed, seeded indices)
DUMP_BYTES = 64 * 10 ** 6    # --dump-outputs writes at most this much in all


def dump_outputs(out_dir, last, dp):
    """What the last timed DataParallelStep.step handed back and left behind, as float32 / float64 .npy files (about 60 MB
    at cfg2): pred [B, T_tgt, V] and hyp [B, T_tgt] as returned, the loss statistics [sum, n_tokens, n_correct, mean,
    1 / n_tokens], the global loss, and a fixed sample of the updated parameters and of the gradients of that step.  A pred
    that would take the total over DUMP_BYTES (--batch > 32) is written as `pred_sample`, a fixed sample of its elements."""
    import numpy as np
    pred, hyp, stats = last
    flat = dp.flat
    idx = torch.from_numpy(np.random.RandomState(0).randint(0, flat.numel, DUMP_SAMPLE)).to(flat.flat.device)
    arrays = {"hyp": hyp.float(), "loss_stats": stats.double(), "global_loss": dp.global_loss().double(),
              "params_sample": flat.flat[idx].float(), "grads_sample": flat.flat_grad[idx].float()}
    room = (DUMP_BYTES - sum(t.numel() * t.element_size() for t in arrays.values()) - 4096) // 4      # float32 elements
    if pred.numel() <= room:
        arrays["pred"] = pred.float()
    else:
        pidx = torch.from_numpy(np.random.RandomState(1).randint(0, pred.numel(), room)).to(pred.device)
        arrays["pred_sample"] = pred.reshape(-1)[pidx].float()
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy())


def run_b200(args, rank, local_rank, world):
    import torch.distributed as dist
    import b200asr
    import importlib
    ops = importlib.import_module(b200asr.__name__ + ".ops")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = b200asr._lib.load(check_device=True)
    if args.precision:
        names = ["linear", "conv", "attn", "conv_wgrad", "attn_bwd"]
        b200asr.precision.set(**dict(zip(names, args.precision.split(","))))
    spec = b200asr.BASELINE_CONFIGS[WORKLOAD]
    cfg, B, T = spec["cfg"], args.batch or spec["batch"], spec["t_src"]
    torch.manual_seed(123456)
    model = b200asr.build_model(cfg).to(dev)
    model.train()
    b200asr.manual_seed(1234 + rank)
    dp = b200asr.DataParallelStep(model, model_size=cfg.dim_input, warmup=4000, k_lr=1.0, min_lr=1e-6,
                                  smoothing=cfg.label_smoothing)
    g = torch.Generator().manual_seed(rank)
    src_h = torch.randn(B, 1, cfg.freq, T, generator=g).pin_memory()
    tgt_h = torch.randint(3, cfg.vocab, (B, cfg.tgt_max_len - 1), generator=g).pin_memory()
    lens = torch.full((B,), T, dtype=torch.int32)
    lens_d = lens.to(dev)
    src_d, tgt_d = src_h.to(dev), tgt_h.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    # ---- device-resident timed region (no instrumentation)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()          # nvidia-smi takes a few 100 ms to produce its first row: start it before the warm-up ...
    for _ in range(args.warmup):
        dp.step(src_d, lens_d, tgt_d)
    barrier()
    sampler.mark()               # ... and keep only the rows sampled from here on (timed + instrumented regions, GPU busy)
    launches0 = lib.b200asr_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        last = dp.step(src_d, lens_d, tgt_d)
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, dp)
    launches = (lib.b200asr_launch_count() - launches0) / args.steps
    ms_dev = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    # ---- forward + loss + backward alone (BASELINE.json's metric names fwd+bwd; `value` above is the whole step incl. the
    #      all-reduce and Adam): single GPU only, the weights do not change so the operand cache stays valid
    fwd_bwd = None
    if world == 1:
        fb_steps = min(args.steps, 10)
        dp.forward_backward(src_d, lens_d, tgt_d)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(fb_steps):
            dp.forward_backward(src_d, lens_d, tgt_d)
        e1.record()
        torch.cuda.synchronize()
        fb_ms = e0.elapsed_time(e1) / fb_steps
        fwd_bwd = {"ms_per_step": fb_ms, "value": B / (fb_ms / 1e3), "unit": "utt/s", "steps": fb_steps,
                   "note": "zero_grad + forward + label-smoothed CE + backward; no all-reduce, no optimizer step"}
    # ---- same steps again with a CUDA-event pair around every C-ABI call (per-kernel-group durations for the roofline);
    #      kept out of `value` because the extra host work per call can starve a ~40 ms step
    prof_steps = min(args.steps, 5)
    ops.profiler.start()
    e0.record()
    for _ in range(prof_steps):
        dp.step(src_d, lens_d, tgt_d)
    e1.record()
    barrier()
    ops.profiler.stop()
    ms_prof = e0.elapsed_time(e1) / prof_steps
    clocks = sampler.stop() if rank == 0 else None
    report = ops.profiler.report()

    # ---- end-to-end through the public API: every step's inputs are copied from pinned host memory (on the prefetcher's side
    #      stream, one batch ahead, as a pin_memory DataLoader would) and the loss is read back by the host, every step
    loss_h = torch.zeros(1).pin_memory()
    pf = b200asr.HostBatchPrefetcher(dev)
    for _ in range(min(2, args.warmup)):
        pf.submit(src_h, tgt_h)
        s, t = pf.take()
        dp.step(s, lens, t)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    pf.submit(src_h, tgt_h)                               # the first batch's copy is inside the timed region too
    for i in range(args.steps):
        s, t = pf.take()
        if i + 1 < args.steps:
            pf.submit(src_h, tgt_h)                       # next batch: copied under this step's kernels
        dp.step(s, lens, t)                               # lengths as the reference's loader hands them over: a CPU tensor
        loss_h.copy_(dp.global_loss().reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()         # the caller reads the loss every step
    e1.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    ms_e2e = max(max_over_ranks(e0.elapsed_time(e1)) / args.steps, 0.0)
    final_loss = float(loss_h.item())

    # ---- the gradient all-reduce alone (N > 1): CUDA events around dp.all_reduce(), max over ranks
    allreduce = None
    if world > 1:
        for _ in range(3):
            dp.all_reduce()
        barrier()
        e0.record()
        for _ in range(10):
            dp.all_reduce()
        e1.record()
        barrier()
        ar_ms = max_over_ranks(e0.elapsed_time(e1)) / 10
        nbytes = dp.flat.flat_grad.numel() * 4
        allreduce = {"ms": ar_ms, "bytes": nbytes, "algbw_gbs": nbytes / ar_ms / 1e6, "busbw_gbs": nbytes / ar_ms / 1e6 * 2 * (world - 1) / world,
                     "note": "one all-reduce(SUM) of the flat fp32 gradient buffer + [sum-loss, n_tokens], timed back to back"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = load_peaks()
    groups = summarize_profile(report, prof_steps, peaks)
    top = next((g for g in groups if g["gflop_per_step"] > 0), groups[0])
    tf32_peak = peaks["bf16_tflops_sustained"] / 2.0       # kind::tf32 runs at half the bf16 rate
    # DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the dominant group come from the tracked ncu
    # summary profiles/ncu_traffic.json (written by tools/ncu_traffic.py from an `ncu --set full` capture of this very
    # command; it records the git revision it was taken at) -- null when that file has no entry for the group
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            tj = json.load(f)
        ent = tj.get("groups", {}).get(top["kernel"])
        if ent:
            traffic, traffic_src = ent["dram_bytes_per_launch"], f"profiles/ncu_traffic.json (git {tj.get('git', '?')}, {ent.get('launches', '?')} launches)"
    except Exception:
        pass
    roof = {"bound": "tensor", "kernel": top["kernel"], "achieved": top["tflops"], "peak": tf32_peak, "unit": "TFLOP/s",
            "frac": top["tflops"] / tf32_peak, "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": f"{peaks['source']} bf16_tflops_sustained/2 (TF32 = half the bf16 tensor rate)",
            "share_of_step": top["share"],
            # 3xTF32 issues three tf32 MMAs per algorithmic product, so `frac` tops out at 1/3 for precision-3 kernels;
            # the tensor-pipe occupancy is frac * mma_per_product (ncu: sm__pipe_tensor_cycles_active, profiles/)
            "mma_per_product": 3 if ops.config.conv_wgrad == 3 else 1,
            "tensor_pipe_frac": top["tflops"] / tf32_peak * (3 if ops.config.conv_wgrad == 3 else 1)}
    # BASELINE.json asks for the achieved fraction of the attention-matmul roofline next to the headline number
    att = [g for g in groups if g["kernel"].startswith("sdpa")]
    att_ms, att_gf = sum(g["ms_per_step"] for g in att), sum(g["gflop_per_step"] for g in att)
    mult = 3 if ops.config.attn in (3, 6) else 1
    attention = {"ms_per_step": att_ms, "gflop_per_step": att_gf, "achieved": att_gf / att_ms if att_ms else 0.0, "unit": "TFLOP/s",
                 "peak": tf32_peak, "frac": (att_gf / att_ms / tf32_peak) if att_ms else 0.0, "mma_per_product": mult,
                 "tensor_pipe_frac": (att_gf / att_ms / tf32_peak * mult) if att_ms else 0.0,
                 "note": ("fused kind::f16 (bf16x3) kernels: QK^T / PV (+ the four backward products, scores recomputed) with masks, "
                          "softmax and dropout on the accumulator in tensor memory; includes the bf16 operand pre-pass")
                 if any(g["kernel"].startswith("sdpa_fused") for g in att) else
                 ("materialised path: batched per-head 3xTF32 GEMMs on the tile engine (QK^T, PV and the four backward products) "
                  "around fp32 softmax / dropout kernels; scores and probabilities stay L2-resident")}
    out = {"metric": METRIC, "value": world * B / (ms_dev / 1e3), "unit": "utt/s", "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32" if not args.precision else "f32(" + args.precision + ")", "data": "synthetic",
           "config": {"workload": WORKLOAD, "per_gpu_batch": B, "global_batch": world * B, "t_src": T, "t_tgt": cfg.tgt_max_len,
                      "dropout": cfg.dropout, "label_smoothing": cfg.label_smoothing,
                      "precision": {"linear": ops.config.linear, "conv": ops.config.conv, "conv_wgrad": ops.config.conv_wgrad,
                                    "attn": ops.config.attn, "attn_bwd": ops.config.attn_bwd,
                                    "legend": "0 = fp32 CUDA cores, 1 = tcgen05 TF32 (RN), 3 = tcgen05 3xTF32 (fp32-grade)"},
                      "step": "zero_grad+fwd+CE+bwd+allreduce+adam", "parallelism": f"dp{world}",
                      "l2": "per-step working set (GBs of activations) >> 126 MB L2; no explicit flush"},
           "e2e": {"value": world * B / (ms_e2e / 1e3), "unit": "utt/s", "h2d_bytes_per_step": world * (src_h.numel() * 4 + tgt_h.numel() * 8),
                   "d2h_bytes_per_step": world * 4, "ms_per_step": ms_e2e, "wall_ms_per_step": wall_ms,
                   "how": "b200asr.HostBatchPrefetcher (pinned host batch copied on a side stream one step ahead, every step) -> "
                          "DataParallelStep.step(src, CPU lengths, tgt) -> loss copied to pinned host memory and the stream "
                          "synchronised, every step"},
           "gpu_launches": launches, "clocks": clocks, "roofline": roof, "attention_roofline": attention, "kernels": groups[:24], "profiled_ms_per_step": ms_prof,
           "final_loss": final_loss}
    if fwd_bwd is not None:
        out["fwd_bwd_only"] = fwd_bwd
    if world == 1 and not args.no_ref_gpu:
        try:
            out["reference_gpu"] = gpu_reference_throughput(dev, B)
        except Exception as e:                      # the reference eager run must never take the product line down
            out["reference_gpu"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    if allreduce is not None:
        out["allreduce"] = allreduce
    if world == 1 and not args.no_cpu:
        ups, mean, threads, kind = cpu_reference_throughput(4, 3, 1)
        out["cpu_baseline"] = {"value": ups, "unit": "utt/s", "cores": threads, "kind": kind,
                               "sample": ("the unmodified reference (oracle/_ref)" if kind == "reference" else "oracle port") +
                                         ": training step, 4 utterances of the cfg2 shape per step, 3 timed steps after 1 warm-up"}
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch override (debug only; the metric uses 32)")
    ap.add_argument("--precision", default="", help="linear,conv,attn[,conv_wgrad[,attn_bwd]] in {fp32,tf32,tf32x3} (default: package default)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip timing the unmodified reference eager on this GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the outputs of the last timed step to DIR/<name>.npy (inputs and weights are seeded, so two "
                         "builds can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
