#!/usr/bin/env python
"""bench.py -- images/sec of the CRNN forward + CTC loss hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c2tf32|c2shape|c1shape] [--impl ours|reference]
                    [--dump-outputs DIR]

One "step" = conv stack -> BiLSTM -> logits -> CTC loss (+gradient, as warp-ctc's forward op computes it)
-> mean + L2, over one synthetic batch.  Default workload = BASELINE.json configs[2] (1xB200 bf16 tcgen05 path,
batch 1024, 32x256): the configuration the north-star targets are quoted on; under torchrun every rank runs the
same per-GPU batch (weak scaling, batch-sharded, no data-path collective for the forward).
Prints ONE JSON line on rank 0.  --dump-outputs DIR: rank 0 also writes what the last timed step returned to its caller
(logits, ctc_costs, ctc_grad, loss) as DIR/<name>.npy; the inputs are seeded, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (per-GPU batch, padded width, description)
    "c3": (1024, 256, "BASELINE configs[2]: bf16 tcgen05 conv+LSTM path, batch 1024, 32x256, fwd+CTC"),
    "c2": (256, 160, "BASELINE configs[1]: fp32-class CRNN fwd+CTC-loss (split-bf16 operands x3, f32 accumulate/elementwise), batch 256, 32x160"),
    "c2tf32": (256, 160, "BASELINE configs[1]: fp32 CRNN fwd+CTC-loss on tcgen05 kind::tf32 operands (f32 accumulate/elementwise), batch 256, 32x160"),
    "c2shape": (256, 160, "BASELINE configs[1] shapes (batch 256, 32x160) on the bf16 path"),
    "c1shape": (32, 100, "BASELINE configs[0] shapes (batch 32, 32x100)"),
}
GFLOP_PER_IMG = lambda W: (12357632 * W - 2097152 + 3145728 * (W // 4 - 1) + 65536 * (W // 4 - 1)) / 1e9   # SURVEY §8(d)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16_burst=d["bf16_tflops"], bf16_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        # median of the upper half: idle samples before/after the region would drag a plain median down
        sm.sort()
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": (float(np.median(load)) if load else None), "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_reference(N, W, steps, warmup, seed=3, run_budget_s=None, n_max=None):
    """The reference's CPU path: the op-for-op fp32 restatement (oracle port) on all host cores.  `run_budget_s`: grow the
    per-step sample from N towards `n_max` (powers of two) as far as warmup+steps steps fit in that many seconds."""
    import torch
    from oracle import crnn_oracle as O
    p32 = O.to_torch(O.init_params(seed, dtype=np.float32), torch.float32)
    data, lab, ll, tsl = O.synth_batch(N, W, seed=seed)
    # "all the host threads it can use": oneDNN on these small convs is fastest well below the core count of a
    # 128-core host, so try a ladder of thread counts once and keep the best (reported as `cores`)
    ncpu = os.cpu_count() or 1
    best = (None, 1e30)
    q = max(1, N // 4)
    for nt in sorted({min(ncpu, c) for c in (8, 16, 32, 64, ncpu)}):
        torch.set_num_threads(nt)
        O.fwd_ctc_fp32(p32, data[:q], lab[:int(ll[:q].sum())], ll[:q], tsl[:q])
        t0 = time.perf_counter()
        O.fwd_ctc_fp32(p32, data[:q], lab[:int(ll[:q].sum())], ll[:q], tsl[:q])
        dt = time.perf_counter() - t0
        if dt < best[1]:
            best = (nt, dt)
    torch.set_num_threads(best[0])
    if run_budget_s is not None and n_max is not None and n_max > N:
        per_step = run_budget_s / float(warmup + steps)
        rate = q / best[1]                                  # images/s seen on the ladder's quarter sample
        n = N
        while n * 2 <= n_max and (n * 2) / rate <= per_step:
            n *= 2
        if n != N:
            N = n
            data, lab, ll, tsl = O.synth_batch(N, W, seed=seed)
    times = []
    loss = None
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        loss, _ = O.fwd_ctc_fp32(p32, data, lab, ll, tsl)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    t = float(np.median(times))
    return dict(value=N / t, ms_per_step=t * 1e3, loss=loss, cores=torch.get_num_threads(), sample_n=N)


def ctc_loss_delta(engine, synthetic, torch, dev, W, n_lines, seeds=(3, 4, 5), compute_dtype="bf16"):
    """GPU path vs the fp64 oracle: total loss (mean CTC NLL + L2) and logits on `n_lines` seeded lines of 32xW per seed."""
    from oracle import crnn_oracle as O
    rows, worst_rel, worst_logit = [], 0.0, 0.0
    for seed in seeds:
        params = synthetic.init_params(seed)
        m = engine.CrnnModel(weight_decay=1e-5, device=dev, compute_dtype=compute_dtype)   # fresh handle: inference mode, untouched parameters
        m.load_params(params)
        data, lab, ll, tsl = synthetic.synth_batch(n_lines, W, seed=seed)
        t_ = lambda a: torch.tensor(a, device=dev)
        lg = m.forward(t_(data), t_(tsl))
        cs, _ = engine.ctc_loss(lg, t_(lab), t_(ll), t_(tsl), max_label_len=int(ll.max()))
        gpu_loss = float(m.total_loss(cs).item())
        p64 = O.to_torch({k: v.astype(np.float64) for k, v in params.items()})
        lo = O.forward(p64, data.astype(np.float64), tsl).numpy()
        co, _ = O.ctc_loss_np(lo, lab, ll, tsl, want_grad=False)
        ref_loss = float(co.mean() + float(O.l2_reg(p64, 1e-5)))
        rel = abs(gpu_loss - ref_loss) / abs(ref_loss)
        lerr = float(np.abs(lg.cpu().numpy() - lo).max() / np.abs(lo).max())
        rows.append({"seed": seed, "gpu": round(gpu_loss, 5), "oracle_fp64": round(ref_loss, 5), "rel": round(rel, 7),
                     "max_logit_err_rel": round(lerr, 6)})
        worst_rel, worst_logit = max(worst_rel, rel), max(worst_logit, lerr)
        del m
    return {"rel": round(worst_rel, 7), "max_logit_err_rel": round(worst_logit, 6), "per_seed": rows, "tolerance": 5e-3 if compute_dtype == "bf16" else 2e-3,
            "within_tolerance": bool(worst_rel <= (5e-3 if compute_dtype == "bf16" else 2e-3)),
            "sample": f"{n_lines} lines of 32x{W} per seed, reference initialisers, fresh inference-mode model vs the fp64 oracle "
                      f"(mean CTC NLL + L2 term; max |logit error| / max |logit|)"}


def run_reference_arm(args, rank):
    """--impl reference: the reference's own CPU implementation of the path (TF1 / warp-ctc cannot be installed: the oracle's
    fp32 torch-CPU port), on the main arm's metric and workload.  Each step is a bounded sample of that workload: as many lines
    of 32xW (a power of two between 32 and the workload's batch) as let warmup+steps steps finish in about 90 s on this host."""
    N_full, W, desc = WORKLOADS[args.workload]
    if rank != 0:
        return
    steps, warmup = max(args.steps, 1), max(args.warmup, 1)
    r = cpu_reference(min(N_full, 32), W, steps, warmup, run_budget_s=90.0, n_max=N_full)
    sample_n = r["sample_n"]
    sample = (f"{sample_n} lines of 32x{W} per step (the workload's batch is {N_full}; CPU throughput per line is flat in the batch "
              f"size), median of {steps} steps after {warmup} warm-up, {r['cores']} torch threads of {os.cpu_count()} host CPUs")
    line = {
        "impl": "reference", "metric": "text-line images/sec (fwd+CTC loss)", "value": r["value"], "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "batch_per_gpu": N_full, "global_batch": N_full * max(args.gpus, 1), "width": W, "T": W // 4 - 1,
                   "reference_sample_per_step": sample_n,
                   "note": "TF1/warp-ctc not installable (py3.12, no network): op-for-op fp32 restatement on torch-CPU, rank 0 only"},
        "cpu_baseline": {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port", "sample": sample,
                         "host_cpus": os.cpu_count()},
        "e2e": {"value": r["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=32, help="lines per CPU-baseline step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the extra training-step measurement")
    ap.add_argument("--no-decode-eq", action="store_true", help="skip the 10k-line decode-equality statistic")
    ap.add_argument("--no-sync-bn", action="store_true", help="N>1: per-replica BatchNorm statistics (round-1 behaviour)")
    ap.add_argument("--no-peer-memory", action="store_true", help="N>1: exchange the BN sums through NCCL instead of peer memory")
    ap.add_argument("--overlap", action="store_true", help="N>1: all-reduce merged gradient buckets on a side stream during the backward "
                                                           "(default: one all-reduce after it; measured faster, profiles/r2_scaling.md)")
    ap.add_argument("--sync-bn-forward", action="store_true", help="N>1: global-batch BN also in the forward-only metric (default: replicas)")
    ap.add_argument("--bucket-mb", type=float, default=8.0, help="N>1: merge announced gradient ranges until this many MB are ready")
    ap.add_argument("--sm-reserve", type=int, default=8, help="N>1 with overlap: SMs the persistent backward kernels leave to the collectives")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    from lstm_ctc_ocr_b200 import engine
    from lstm_ctc_ocr_b200._lib import c_int, check
    from lstm_ctc_ocr_b200.lib.networks.factory import get_network
    from lstm_ctc_ocr_b200.session import Session
    from lstm_ctc_ocr_b200 import synthetic

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    if world > 1:
        if args.overlap:
            os.environ.setdefault("NCCL_MAX_NCHANNELS", str(max(args.sm_reserve, 1)))     # the overlapped collectives fit the reserved SMs
        dist.init_process_group("nccl", device_id=dev)
    N, W, desc = WORKLOADS[args.workload]
    T = W // 4 - 1
    K, Wm = args.steps, args.warmup
    peaks = load_peaks()

    # ---- model with reference initialisers (random init; no checkpoints offline), identical on every rank
    f32_path = args.workload in ("c2", "c2tf32")
    cdt = {"c2": "f32", "c2tf32": "tf32"}.get(args.workload, "bf16")     # engine.CrnnModel(compute_dtype=...)
    model = engine.CrnnModel(weight_decay=1e-5, device=dev, compute_dtype=cdt)
    model.load_params(synthetic.init_params(3))
    if f32_path:
        args.no_train = True            # the f32-class path is forward + CTC only (BASELINE configs[1])
    # ---- N > 1: the batch is sharded over ranks; BatchNorm statistics are taken over the GLOBAL batch (exchanged inside the BN
    # finalize kernel over NVLink peer memory, csrc/peer.cu) so that "whole-box batch" means what it means on one device
    dp = None
    if world > 1:
        from lstm_ctc_ocr_b200 import parallel
        dp = parallel.DataParallel(model, sync_bn=not args.no_sync_bn, overlap=args.overlap, peer_memory=not args.no_peer_memory,
                                   min_bucket_bytes=int(args.bucket_mb * (1 << 20)), sm_reserve=args.sm_reserve)
        # forward + CTC metric: independent replicas, each normalising with the statistics of ITS batch of 1024 (what N reference
        # processes would do; decode is "replicas only", SURVEY 8(e)).  The training step below switches to GLOBAL-batch statistics.
        train_sync_bn = dp.sync_bn
        if not args.sync_bn_forward:
            dp.set_sync_bn(False)

    # ---- rotating set of distinct input batches > L2 (8 x 33.5 MB at c3), resident in HBM
    nrot = max(2, int(np.ceil(160e6 / (N * W * 32 * 4))))
    batches = []
    for i in range(nrot):
        data, lab, ll, tsl = synthetic.synth_batch(N, W, seed=3 + 1000 * rank + i)
        batches.append((torch.tensor(data, device=dev), torch.tensor(lab, device=dev), torch.tensor(ll, device=dev),
                        torch.tensor(tsl, device=dev), int(ll.max()), (data, lab, ll, tsl)))
    logits = torch.empty((T, N, 64), dtype=torch.float32, device=dev)
    costs = torch.empty(N, dtype=torch.float32, device=dev)
    grad = torch.empty_like(logits)

    def step(i):
        d, lab, ll, tsl, mll, _ = batches[i % nrot]
        model.forward(d, tsl, out=logits)
        engine.ctc_loss(logits, lab, ll, tsl, want_grad=True, grad_scale=1.0 / N, max_label_len=mll, costs=costs, grad=grad)
        return model.total_loss(costs)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for i in range(Wm):
        loss = step(i)
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    # ---- timed region: K steps, CUDA events on the launching stream, per-stage events inside
    check(model.lib.crnn_profile_begin(model.handle, K))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctc_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    sync_all()
    e0.record()
    for i in range(K):
        d, lab, ll, tsl, mll, _ = batches[i % nrot]
        model.forward(d, tsl, out=logits)
        ctc_ev[i][0].record()
        engine.ctc_loss(logits, lab, ll, tsl, want_grad=True, grad_scale=1.0 / N, max_label_len=mll, costs=costs, grad=grad)
        ctc_ev[i][1].record()
        loss = model.total_loss(costs)
    e1.record()
    sync_all()
    if args.dump_outputs and rank == 0:
        # read before the sections below reuse these buffers: ~33 MB at c3, all f32
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in (("logits", logits), ("ctc_costs", costs), ("ctc_grad", grad), ("loss", loss)):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.cpu().numpy())
    ms_total = e0.elapsed_time(e1)
    loss_val = float(loss.item())
    nst = model.lib.crnn_profile_num_stages()
    buf = (np.zeros((K, nst), dtype=np.float32))
    nf = c_int()
    check(model.lib.crnn_profile_read(model.handle, buf.ctypes.data, nf))
    stage_ms = buf[:nf.value].mean(axis=0) if nf.value > 0 else np.zeros(nst, np.float32)
    stage_names = [model.lib.crnn_profile_stage_name(i).decode() for i in range(nst)]
    ctc_ms = float(np.mean([a.elapsed_time(b) for a, b in ctc_ev]))

    # ---- e2e: the reference-facing call (Session.run on HOST numpy buffers; H2D + D2H inside the timed region), three feeds:
    #   feeder          fresh batch every step, produced by the PrefetchFeeder's worker processes straight into page-locked ring
    #                   slots (lib/lstm/utils/gen.py; replaces GeneratorEnqueuer + Queue, reference gen.py:112-128) -> DMA in place,
    #                   chunked and overlapped with the conv front end (crnn_forward_host).  THE HEADLINE e2e.
    #   fresh_pageable  a brand-new pageable numpy array every step, as the reference's solver builds it (train.py:119-125):
    #                   host copy into pinned staging, then copy-then-compute
    #   refed_buffers   round 1's best case: the same few host buffers fed again and again (page-locked in place on re-sighting)
    from lstm_ctc_ocr_b200.lib.lstm.utils import gen as datagen
    net = get_network("LSTM_train")
    sess = Session(device=dev)
    sess._engines[id(net)] = model            # same weights / same engine instance
    loss_h, _ = net.build_loss()
    Ke = max(3, min(K, 10))

    def run_on(data, lab, ll, tsl):
        return sess.run(loss_h, feed_dict={net.data: data, net.labels: lab, net.time_step_len: tsl, net.labels_len: ll, net.keep_prob: 0.5})

    def timed(fn, n):
        sync_all()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for i in range(n):
            out = fn(i)
        f1.record()
        sync_all()
        return f0.elapsed_time(f1), out

    e2e_var = {}
    # (a) feeder
    nwork = int(os.environ.get("CRNN_BENCH_FEED_WORKERS", "8"))
    arg_fn = lambda k: dict(k=k, batch_size=N, render=False, seed=3 + 1000 * rank, rank=0, world=1, width=W, cache=4)
    feeder = datagen.PrefetchFeeder(arg_fn, num_workers=nwork, depth=4, max_width=W, batch_size=N, keep=2,
                                    warm=[arg_fn(k) for k in range(4)])      # every producer draws its 4 cached batches at start-up
    try:
        if not os.environ.get("CRNN_BENCH_NO_DEVICE_PREFETCH"):
            sess.attach_feeder(feeder)        # the next ring slot's H2D copy overlaps the current step (one 33.6 MB copy per step either way)

        def feed_step(i):
            view, lab, ll, tsl = next(feeder)
            return run_on(view, np.asarray(lab, np.int32), np.asarray(ll, np.int32), np.asarray(tsl, np.int32))
        for i in range(max(16, 8 * nwork)):   # producers come up (caches filled by the pool initializer) and touch every ring slot once
            feed_step(i)
        feed_path = sess.last_feed_path
        ms_feed, e2e_loss = timed(feed_step, Ke)
        h2d_b, d2h_b = int(sess.h2d_bytes), int(sess.d2h_bytes)
        feed_path = sess.last_feed_path
        prefetch_hits = int(sess.ahead_hits)
        # the same feeder WITHOUT the device prefetch: every step's H2D copy (4 chunks, overlapped with conv1..conv3_2) inside its own step
        sess.attach_feeder(None)
        for i in range(4):
            feed_step(i)
        ms_feed_instep, _ = timed(feed_step, Ke)
    finally:
        sess.attach_feeder(None)
        feeder.close()
    # (b) fresh pageable array every step
    fresh = [np.array(batches[i % nrot][5][0]) for i in range(Ke + 2)]
    try:
        run_on(fresh[0], *batches[0][5][1:]); run_on(fresh[1], *batches[1 % nrot][5][1:])
        ms_fresh, l_fresh = timed(lambda i: run_on(fresh[i + 2], *batches[(i + 2) % nrot][5][1:]), Ke)
        fresh_path = sess.last_feed_path + (" (host-thread pool -> page-locked staging, pipelined with the DMA: crnn_forward_pageable)"
                                            if sess.h2d_chunks > 1 and sess.pageable_pool else "")
        # same inputs through the resident-input forward: the side statistic must not be the only check of this path
        ref_l = float(model.total_loss(engine.ctc_loss(model.forward(batches[(Ke + 1) % nrot][0], batches[(Ke + 1) % nrot][3]), batches[(Ke + 1) % nrot][1],
                                                       batches[(Ke + 1) % nrot][2], batches[(Ke + 1) % nrot][3],
                                                       max_label_len=batches[(Ke + 1) % nrot][4])[0]).item())
        if not abs(float(l_fresh) - ref_l) <= 2e-3 * abs(ref_l):
            fresh_path += f" LOSS MISMATCH {float(l_fresh)} vs {ref_l}"
    except Exception as e:                    # never lose the bench line over a variant
        ms_fresh, fresh_path = float("inf"), "failed: " + repr(e)[:200]
    del fresh
    # (c) the same host buffers re-fed
    for i in range(max(3, 3 * nrot)):
        run_on(*batches[i % nrot][5])
    ms_refed, _ = timed(lambda i: run_on(*batches[i % nrot][5]), Ke)
    ms_e2e = ms_feed
    clocks = sampler.stop() if rank == 0 else None

    # ---- BASELINE configs[4] companion: full training step (fwd + CTC + backward + [NCCL grad all-reduce] + clip + Adam)
    ms_train = None
    ms_fwd_sync = None
    if dp is not None and train_sync_bn:
        dp.set_sync_bn(True)
        if not args.sync_bn_forward:
            # the same forward + CTC step with BatchNorm over the GLOBAL batch (2 x 8 KB exchanged inside the BN finalize kernel)
            for i in range(3):
                step(i)
            sync_all()
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0.record()
            for i in range(K):
                step(i)
            h1.record()
            sync_all()
            ms_fwd_sync = h0.elapsed_time(h1) / K
    if not args.no_train:
        model.set_training(True)
        Kt = max(3, min(K, 10))

        def train_step(i, stepno):
            d, lab, ll, tsl, mll, _ = batches[i % nrot]
            model.forward(d, tsl, out=logits)
            engine.ctc_loss(logits, lab, ll, tsl, want_grad=True, grad_scale=1.0 / N, max_label_len=mll, costs=costs, grad=grad)
            model.backward(d, tsl, grad)        # N>1: announces 7 gradient buckets; each is all-reduced on a side stream meanwhile
            if dp is not None:
                dp.step(1e-4, stepno, clip=10.0)
            else:
                model.clip_adam_step(lr=1e-4, step=stepno, clip=10.0)
        for i in range(3):
            train_step(i, i + 1)
        sync_all()
        check(model.lib.crnn_profile_begin(model.handle, Kt))
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for i in range(Kt):
            train_step(i, 4 + i)
        g1.record()
        sync_all()
        ms_train = g0.elapsed_time(g1) / Kt
        nb = model.lib.crnn_profile_bwd_num_stages()
        bbuf = np.zeros((Kt, nb), dtype=np.float32)
        nfb = c_int()
        check(model.lib.crnn_profile_bwd_read(model.handle, bbuf.ctypes.data, nfb))
        bwd_stage_ms = {model.lib.crnn_profile_bwd_stage_name(i).decode(): round(float(bbuf[:nfb.value, i].mean()), 4) for i in range(nb)}
        fbuf = np.zeros((Kt, nst), dtype=np.float32)
        check(model.lib.crnn_profile_read(model.handle, fbuf.ctypes.data, nfb))
        bwd_stage_ms["forward_total(train mode)"] = round(float(fbuf[:nfb.value].sum(axis=1).mean()), 4)
        fwd_train_stage_ms = {n_: round(float(v_), 4) for n_, v_ in zip(stage_names, fbuf[:nfb.value].mean(axis=0))} if nfb.value > 0 else {}

    # ---- max over ranks
    if world > 1:
        t = torch.tensor([ms_total, ms_e2e, ms_train or 0.0, ms_fresh, ms_refed, ms_fwd_sync or 0.0], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e = float(t[0]), float(t[1])
        ms_train = float(t[2]) if ms_train is not None else None
        ms_fresh, ms_refed = float(t[3]), float(t[4])
        ms_fwd_sync = float(t[5]) if ms_fwd_sync is not None else None
    ms_step = ms_total / K
    value = world * N / (ms_step / 1e3)
    e2e_value = world * N / (ms_e2e / Ke / 1e3)

    if rank == 0:
        # dominant kernel = the stage with the largest share of the step
        flops = {"conv2_pool2": 2.0 * N * (W // 2) * 16 * 576 * 128, "conv3_1": 2.0 * N * (W // 4) * 8 * 1152 * 256,
                 "conv3_2_pool": 2.0 * N * (W // 4) * 8 * 2304 * 256, "conv4_1_gemm": 2.0 * N * (W // 4) * 4 * 2304 * 512,
                 "conv4_2_gemm": 2.0 * N * (W // 4) * 4 * 4608 * 512, "conv5": 2.0 * N * T * 2048 * 512,
                 "lstm_xproj": 2.0 * N * T * 512 * 2048, "lstm_recurrence": 2.0 * N * T * 256 * 1024 * 2, "logits": 2.0 * N * T * 512 * 64,
                 "conv1_pool1": 2.0 * N * W * 32 * 9 * 64}
        stages = {n: {"ms": round(float(m), 4), "share": round(float(m) / ms_step, 4),
                      **({"tflops": round(flops[n] / (float(m) * 1e-3) / 1e12, 1)} if n in flops and m > 0 else {})}
                  for n, m in zip(stage_names, stage_ms)}
        ctc_bytes = 2 * T * N * 64 * 4 + 4 * (int(batches[0][1].numel()) + 2 * N)
        stages["ctc_loss_grad"] = {"ms": round(ctc_ms, 4), "share": round(ctc_ms / ms_step, 4),
                                   "gbs": round(ctc_bytes / (ctc_ms * 1e-3) / 1e9, 1),
                                   "hbm_frac": round(ctc_bytes / (ctc_ms * 1e-3) / 1e9 / peaks["hbm"], 3)}
        dom = max((n for n in stage_names if n in flops and n != "conv1_pool1" and n != "lstm_recurrence"),
                  key=lambda n: stages[n]["ms"])
        ach = flops[dom] / (max(stages[dom]["ms"], 1e-9) * 1e-3) / 1e12
        traffic = None
        tp = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
        if os.path.exists(tp) and args.workload == "c3":
            traffic = json.load(open(tp))["kernels"].get(dom, {}).get("traffic_bytes")
        roofline = {"kernel": f"gemm_kernel<{dom}>", "bound": "tensor", "achieved": round(ach, 1), "peak": peaks["bf16_sustained"],
                    "unit": "TFLOP/s", "frac": round(ach / peaks["bf16_sustained"], 3), "traffic": traffic,
                    "traffic_note": "DRAM read+write bytes of one launch from the committed ncu --set full capture (profiles/r2_ncu_traffic.json); "
                                    "algorithmic bytes of conv4_2 = 268 MB in + 4.7 MB weights + 268 MB out",
                    "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['src']}); kernel timed inside a long step",
                    "whole_step_tflops": round(N * GFLOP_PER_IMG(W) / ms_step, 1),
                    # the same achieved figure against the BURST cuBLAS number of the same file (a frac above 1 against the sustained
                    # one means: this kernel, inside the step, runs faster than cuBLAS does in a 4 s back-to-back loop on this box)
                    "peak_burst": peaks["bf16_burst"], "frac_of_burst": round(ach / peaks["bf16_burst"], 3)}
        line = {
            "metric": "text-line images/sec (fwd+CTC loss)", "value": round(value, 1), "unit": "images/s", "n_gpus": world,
            "steps": K, "warmup": Wm, "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": {"f32": "f32 (bf16x3 split operands, f32 accumulate)", "tf32": "tf32 (kind::tf32 operands, f32 accumulate)"}.get(cdt, "bf16"),
            "data": "synthetic",
            "config": {"workload": desc, "batch_per_gpu": N, "global_batch": N * world, "width": W, "T": T,
                       "parallelism": (f"dp{world}: batch sharded over ranks; BatchNorm over the GLOBAL batch -- 2 exchanges of 8 KB per forward, "
                                       f"{'fused into the BN finalize kernel over NVLink peer memory' if (dp is not None and dp.peer) else 'NCCL all-reduce'}"
                                       if (dp is not None and args.sync_bn_forward and not args.no_sync_bn)
                                       else f"dp{world}: independent replicas for forward + CTC (each BatchNorm over its own batch of {N}); "
                                            f"the train_step entry shards ONE global batch (global-batch BN, gradient all-reduce)"),
                       "l2": f"rotating {nrot} distinct input batches ({nrot * N * W * 32 * 4 / 1e6:.0f} MB > 126 MB L2); "
                             f"per-step activation traffic ~2.5 GB"},
            "loss": round(loss_val, 5),
            "e2e": {"value": round(e2e_value, 1), "unit": "images/s", "h2d_bytes_per_step": h2d_b,
                    "d2h_bytes_per_step": d2h_b, "steps": Ke, "api": "Session.run(loss, feed_dict=host numpy)",
                    "feed": f"PrefetchFeeder: a fresh batch every step, written by {nwork} producer processes into page-locked "
                            f"shared-memory ring slots, DMA'd in place ({feed_path})",
                    "pipelining": ("Session.attach_feeder: the H2D copy of step i+1's ring slot (and its integer feeds) is issued on a side stream once step i's "
                                   f"kernels are enqueued, step i+1 waits for it on the GPU; every timed step issues one {h2d_b / 1e6:.1f} MB copy and consumes one "
                                   f"(prefetch hits so far: {prefetch_hits}); the loss is read back synchronously every step"),
                    "loss": float(e2e_loss),
                    "variants": {
                        "feeder_copy_inside_own_step": {"value": round(world * N / (ms_feed_instep / Ke / 1e3), 1),
                                                        "what": "same feeder without the device prefetch: the chunked H2D copy overlaps only its own step's conv front end (the r2 mid-round e2e)"},
                        "fresh_pageable_array_every_step": {"value": round(world * N / (ms_fresh / Ke / 1e3), 1), "path": fresh_path,
                                                            "what": "np.array(...) built per step as reference train.py:119-125 does; staged through pinned memory"},
                        "refed_host_buffers": {"value": round(world * N / (ms_refed / Ke / 1e3), 1),
                                               "what": "round-1 e2e: the same host buffers re-fed (page-locked in place on re-sighting)"}}},
            "gpu_launches": K * 16,      # per step: conv1, 8 tcgen05 GEMMs, 2x(bn finalize + apply), persistent LSTM, CTC, loss
            "roofline": roofline, "stages": stages, "clocks": clocks,
        }
        if f32_path:
            # no per-stage events on this path: the whole step against the tensor peak of a 3-product contraction
            wt = N * GFLOP_PER_IMG(W) / ms_step
            div = 2.0 if cdt == "tf32" else 3.0
            line["roofline"] = {"kernel": ("whole step (gemm_kernel kind::tf32 + f32 elementwise passes + per-step LSTM launches)" if cdt == "tf32" else
                                           "whole step (gemm_kernel x3 products + f32 elementwise passes + per-step LSTM launches)"), "bound": "tensor",
                                "achieved": round(wt, 1), "peak": round(peaks["bf16_sustained"] / div, 1), "unit": "TFLOP/s",
                                "frac": round(wt / (peaks["bf16_sustained"] / div), 3), "traffic": None,
                                "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained / 2 (kind::tf32 issues at half the kind::f16 rate; no tf32 figure is measured)"
                                                if cdt == "tf32" else
                                                "MEASURED_PEAKS.json bf16_tflops_sustained / 3 (each fp32-class product is three bf16 MMAs); "
                                                "achieved counts the ALGORITHMIC flops once")}
            line.pop("stages", None)
            line["gpu_launches"] = K * (1 + 2 * 6 + 4 + 2 + 2 * T + 4)
        if ms_fwd_sync is not None:
            line["global_batch_bn_forward"] = {"ms_per_step": round(ms_fwd_sync, 4), "images_per_s": round(world * N / (ms_fwd_sync / 1e3), 1),
                                               "what": "the same forward + CTC step with BatchNorm statistics over the GLOBAL batch "
                                                       f"({world * N} lines): two 8 KB exchanges per step inside the BN finalize kernel "
                                                       f"({'NVLink peer memory' if dp.peer else 'NCCL callback'}); the extra time is the wait for the slowest rank"}
        if ms_train is not None:
            line["train_step"] = {"ms_per_step": round(ms_train, 4), "images_per_s": round(world * N / (ms_train / 1e3), 1),
                                  "what": "fwd + CTC loss/grad + backward + " + ((f"NCCL all-reduce(28.6 MB f32) in buckets >= {args.bucket_mb:g} MB overlapped with the backward ({args.sm_reserve} SMs reserved) + " if args.overlap else "one NCCL all-reduce(28.6 MB f32) after the backward + ") +
                                          (("global-batch BatchNorm (sums exchanged inside the BN kernels over NVLink peer memory) fwd/bwd + " if (dp is not None and dp.peer)
                                            else "global-batch BatchNorm (sums through an NCCL all-reduce callback) fwd/bwd + ") if not args.no_sync_bn else "") if world > 1 else "") +
                                          "global-norm clip + Adam (BASELINE configs[4] per-GPU shape)",
                                  "stages_ms": bwd_stage_ms, "forward_stages_train_mode_ms": fwd_train_stage_ms}
        if world == 1 and not args.no_cpu_baseline:
            sn = args.cpu_sample
            r = cpu_reference(sn, W, steps=8, warmup=2)
            line["cpu_baseline"] = {"value": round(r["value"], 2), "unit": "images/s", "cores": r["cores"], "kind": "port",
                                    "sample": f"{sn} lines of 32x{W} per step (same shapes, fp32 torch-CPU restatement), median of 8"}
            line["cpu_baseline"]["host_cpus"] = os.cpu_count()
            line["cpu_baseline"]["threads_note"] = "cores = torch threads that ran fastest on this host (ladder 8/16/32/64/all); host_cpus = os.cpu_count()"
            # BASELINE metric, second half ("CTC-loss delta vs ref"): a FRESH inference-mode model with the reference initialisers
            # (VERDICT r1 weak #1: the round-1 figure was taken on a model that had already run 13 Adam steps) against the fp64
            # oracle on the same seeded 32x256 samples, three seeds.
            try:
                line["ctc_loss_delta"] = ctc_loss_delta(engine, synthetic, torch, dev, W, sn, compute_dtype=cdt)
            except Exception as e:      # never lose the bench line over the side statistic
                line["ctc_loss_delta"] = {"error": repr(e)[:300]}
            # BASELINE configs[3] / north-star: greedy-decode sequence equality with the oracle on 10k rendered lines, through the model
            # (images -> Session.run(dense_decoded)), bucketed batches of 512; the oracle's decode is a committed fixture
            # (tests/golden/make_decode10k.py), so no CPU forward runs here.  Filtered count reported, nothing hidden.
            if not args.no_decode_eq and os.path.exists(os.path.join(ROOT, "tests", "golden", "decode10k_oracle.npz")):
                try:
                    import importlib.util
                    spec = importlib.util.spec_from_file_location("t10k", os.path.join(ROOT, "tests", "test_gpu_decode10k.py"))
                    t10k = importlib.util.module_from_spec(spec)
                    spec.loader.exec_module(t10k)
                    st = t10k.run_decode10k(cdt, device=dev)
                    st.pop("per_width", None)
                    line["decode_equality"] = st
                except Exception as e:
                    line["decode_equality"] = {"error": repr(e)[:300]}
        print(json.dumps(line), flush=True)
    if world > 1:
        if dp is not None:
            perr = dp.peer_error() if dp.peer else 0
            if perr and rank == 0:
                sys.stderr.write("WARNING: a peer-memory exchange timed out\n")
            dp.close()
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
