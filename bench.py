#!/usr/bin/env python
"""bench.py -- the hot path's benchmark (contract: task brief §④).

One "step" = one DIR training step on one synthetic batch per GPU:
  ResNet-50 forward (train-mode BN) -> FDS.smooth (live tables, epoch >= 2 state)
  -> 2048->1 regressor -> LDS-weighted L1 loss -> backward -> [NCCL grad all-reduce]
  -> Adam, all through this repo's public (reference-shaped) API.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B]   # our arm (N>1: under torchrun)
  python bench.py ... --dump-outputs DIR                            # + what the last timed step computed, DIR/*.npy
  python bench.py --impl reference ...                              # the CPU arm (oracle port, host cores)

Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "imbalanced-regression_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

# BASELINE.json configs[2], the configuration the metric is quoted on (SURVEY.md section 8d, C3)
WORKLOAD = "IMDB-WIKI-DIR ResNet-50 + FDS (feature_dim 2048, bucket_num 100, bucket_start 0, gaussian ks5 sigma2) + " \
           "LDS (sqrt_inv, gaussian ks5 sigma2) weighted L1, bf16, batch 256/GPU, synthetic 224x224, Adam; labels drawn " \
           "from the IMDB-WIKI train age histogram (ages 0-186, > 99 folded into the edge bin)"
BUCKET_NUM, BUCKET_START = 100, 0
FWD_GFLOP_PER_IMG = 8.174          # SURVEY.md §8(d)
FWDBWD_GFLOP_PER_IMG = 24.29
SPEC_BF16_TFLOPS = 2250.0          # B200 dense bf16, nominal (B200_PROFILING.md)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_burst=d["bf16_tflops"], bf16_sustained=d["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    QUERY = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown," \
            "clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


_IMDB_AGES = None


def synthetic_labels(n, seed):
    """n labels drawn (with replacement) from the real IMDB-WIKI training label column (191 509 ages, 0..186: the
    fixture tests/golden/lds.npz carries it), so the timed step sees the reference's label distribution including the
    ages > bucket_num - 1 that FDS folds into the edge bin; a gamma-shaped stand-in when the fixture is absent."""
    global _IMDB_AGES
    rng = np.random.RandomState(seed)
    if _IMDB_AGES is None:
        path = os.path.join(ROOT, "tests", "golden", "lds.npz")
        try:
            _IMDB_AGES = np.load(path)["imdb_wiki_labels"].astype(np.float32)
        except Exception:  # noqa: BLE001
            _IMDB_AGES = np.zeros(0, np.float32)
    if _IMDB_AGES.size:
        return _IMDB_AGES[rng.randint(0, _IMDB_AGES.size, size=n)].copy()
    return np.clip(np.round(rng.gamma(shape=6.0, scale=6.5, size=n)), 0, 186).astype(np.float32)


# ----------------------------------------------------------------------------- CPU arm
def cpu_threads():
    """Host threads for the CPU arm: all cores up to 32 -- beyond that torch's CPU conv/BN kernels on a small batch
    slow down badly (measured on the 128-thread B200 host: 0.05-0.5 img/s with 128 threads)."""
    return max(1, min(os.cpu_count() or 1, 32))


def _epoch_features(n=12208, seed=7):
    rng = np.random.RandomState(seed)
    lab = synthetic_labels(n, seed)
    feats = np.maximum(rng.randn(n, 2048).astype(np.float32) * (1.0 + 0.01 * lab[:, None]) + 0.5, 0).astype(np.float32)
    return feats, lab


class _CpuArm:
    """The reference's own modules (oracle/_ref, oracle/ref_step.py) when installed, else the port
    (oracle/train_ref.py); same step either way: ResNet-50 fwd (train-mode BN) -> FDS.smooth (epoch >= 2 tables) ->
    regressor -> LDS-weighted L1 -> backward -> Adam, fp32 on the host cores."""

    def __init__(self):
        from oracle import ref_step
        torch.set_num_threads(cpu_threads())
        feats, lab = _epoch_features()
        self.feats, self.lab = feats, lab
        if ref_step.available():
            self.kind = "reference"
            self.tr = ref_step.ReferenceTrainer(bucket_num=BUCKET_NUM, bucket_start=BUCKET_START, epoch_features=feats,
                                                epoch_labels=lab)
            self.what = "the reference's own resnet.py / fds.py / loss.py (oracle/_ref), torch fp32 CPU kernels"
        else:
            from oracle.train_ref import RefTrainer
            self.kind = "port"
            g = torch.Generator().manual_seed(0)
            nb = BUCKET_NUM - BUCKET_START
            tables = (torch.randn(nb, 2048, generator=g) * .1 + .5, torch.rand(nb, 2048, generator=g) + .5,
                      torch.randn(nb, 2048, generator=g) * .1 + .5, torch.rand(nb, 2048, generator=g) + .5)
            self.tr = RefTrainer(bucket_num=BUCKET_NUM, bucket_start=BUCKET_START, fds_tables=tables)
            self.what = "oracle/train_ref.py (port: oracle/_ref not installed), torch fp32 CPU kernels"

    def batch(self, bs):
        g = torch.Generator().manual_seed(0)
        x = torch.randn(bs, 3, 224, 224, generator=g)
        t = torch.from_numpy(synthetic_labels(bs, 1)).reshape(bs, 1)
        return x, t, torch.ones(bs, 1)

    def fds_ms(self):
        """SURVEY 8(d): the FDS stages on the host CPU, `update_running_stats` over an AgeDB-sized feature matrix
        (N = 12 208 x 2048) and `smooth` on one batch of 256, median of 3, ms; never fails the bench."""
        try:
            if self.kind == "reference":
                return self.tr.fds_timings(self.feats, self.lab)
            from oracle import dir_oracle as O
            st = O.FDSState(2048, BUCKET_NUM, BUCKET_START, kernel="gaussian", ks=5, sigma=2)
            st.update_last_epoch_stats(0)
            upd, smo = [], []
            for ep in range(3):
                t0 = time.perf_counter()
                st.update_running_stats(self.feats, self.lab, ep)
                upd.append(time.perf_counter() - t0)
                st.update_last_epoch_stats(ep + 1)
            for _ in range(3):
                t0 = time.perf_counter()
                st.smooth(self.feats[:256], self.lab[:256], 3)
                smo.append(time.perf_counter() - t0)
            return {"update_running_stats_ms": round(1e3 * sorted(upd)[1], 2), "smooth_b256_ms": round(1e3 * sorted(smo)[1], 2),
                    "rows": 12208, "impl": "oracle/dir_oracle.py (numpy port)"}
        except Exception as e:  # noqa: BLE001
            return {"error": repr(e)[:200]}


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the step on the box's host cores; each step is a
    bounded sample (--cpu-batch images) of the 256-image workload so that K + W steps end within minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = _CpuArm()
    bs = args.cpu_batch
    x, t, w = arm.batch(bs)
    for _ in range(args.warmup):
        arm.tr.step(x, t, w)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        arm.tr.step(x, t, w)
    dt = time.perf_counter() - t0
    val = bs * args.steps / dt
    sample = f"{args.steps} steps of batch {bs} of the batch-256 workload ({arm.what}, {torch.get_num_threads()} threads)"
    out = {"impl": "reference", "metric": "images/sec", "value": val, "unit": "images/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": WORKLOAD, "sample": sample},
           "cpu_baseline": {"value": val, "unit": "images/s", "cores": torch.get_num_threads(), "kind": arm.kind,
                            "sample": sample, "fds_ms": arm.fds_ms()},
           "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


def cpu_baseline_sample(seconds_budget=20.0, bs=16):
    arm = _CpuArm()
    x, t, w = arm.batch(bs)
    arm.tr.step(x, t, w)
    n, t0 = 0, time.perf_counter()
    while n < 2 or (time.perf_counter() - t0 < seconds_budget and n < 12):
        arm.tr.step(x, t, w)
        n += 1
    dt = time.perf_counter() - t0
    return {"value": bs * n / dt, "unit": "images/s", "cores": torch.get_num_threads(), "kind": arm.kind,
            "sample": f"{n} steps of batch {bs} after 1 warm-up ({arm.what})", "fds_ms": arm.fds_ms()}


# ----------------------------------------------------------------------------- GPU arm
def build_training_state(args, device, rank, world):
    from resnet import resnet50
    from optim import FusedAdam
    from parallel import DataParallel
    from datasets import lds_prepare_weights
    torch.manual_seed(0)
    model = resnet50(fds=True, bucket_num=BUCKET_NUM, bucket_start=BUCKET_START, start_update=0, start_smooth=1,
                     kernel="gaussian", ks=5, sigma=2, momentum=0.9).to(device)
    model = DataParallel(model)
    model.broadcast_parameters()
    model.train()
    fds = model.module.FDS
    # bring FDS to its epoch >= 2 state through the module's own epoch-end path (train.py:269-281 order): every rank
    # streams ITS shard of a synthetic epoch of features into the accumulators, finish_epoch_stats all-reduces
    # (count, sum, sum of squares) and the edge flags across the ranks -> identical tables everywhere
    n_ep = 12208
    ep_labels = torch.from_numpy(synthetic_labels(n_ep, 7)).to(device)
    gen = torch.Generator(device=device).manual_seed(123)          # same stream on every rank
    for epoch in (0, 1):
        feats = torch.relu(torch.randn(n_ep, 2048, device=device, generator=gen) * (1.0 + 0.01 * ep_labels[:, None])
                           + 0.5)
        fds.begin_epoch_stats(ep_labels[rank::world])
        for i in range(rank, n_ep, world * 4096):                  # this rank's rows, a few chunks
            sl = slice(i, min(i + world * 4096, n_ep), world)
            fds.accumulate_batch(feats[sl], ep_labels[sl])
        fds.update_last_epoch_stats(epoch)
        fds.finish_epoch_stats(epoch)
    fds.update_last_epoch_stats(2)
    # LDS weights from the whole (synthetic) training-label column: sqrt_inv + gaussian ks5 sigma2
    w_all = lds_prepare_weights(ep_labels.cpu().numpy(), "sqrt_inv", lds=True, lds_kernel="gaussian", lds_ks=5,
                                lds_sigma=2)
    opt = FusedAdam(model.parameters(), lr=1e-3, grad_scale=1.0 / world)
    return model, opt, ep_labels, w_all


def make_batches(args, device, rank, ep_labels, w_all, pinned):
    """A few distinct synthetic batches (x fp32 NCHW, targets, LDS weights)."""
    g = torch.Generator().manual_seed(1000 + rank)
    batches = []
    for i in range(args.num_batches):
        idx = torch.randint(0, ep_labels.numel(), (args.batch,), generator=g)
        x = torch.randn(args.batch, 3, 224, 224, generator=g)
        t = ep_labels.cpu()[idx].reshape(-1, 1).clone()
        w = w_all.cpu()[idx].reshape(-1, 1).clone()
        if pinned:
            batches.append(tuple(a.pin_memory() for a in (x, t, w)))
        else:
            batches.append(tuple(a.to(device) for a in (x, t, w)))
    return batches


def train_step(model, opt, x, t, w, epoch=2):
    from loss import weighted_l1_loss
    outputs, encoding = model(x, t, epoch)
    loss = weighted_l1_loss(outputs, t, w)
    opt.zero_grad()
    loss.backward()
    model.reduce_gradients()
    opt.step()
    return loss, outputs, encoding


DUMP_SAMPLE = 1 << 22      # parameters / gradients written by --dump-outputs: 16 MB each as float32


def dump_outputs(out_dir, loss, outputs, encoding, net):
    """--dump-outputs: what one training step hands back -- the loss, the predictions, the encoding the forward
    returns, the BatchNorm running statistics it updated, and the same fixed, seeded sample of the updated parameters
    and of their gradients -- as float32 DIR/<name>.npy (~34 MB in all), so that two builds can be compared output for
    output."""
    os.makedirs(out_dir, exist_ok=True)
    flat = net.flat_parameters()
    idx = np.random.default_rng(0).choice(flat.numel(), size=min(DUMP_SAMPLE, flat.numel()), replace=False)
    idx = torch.from_numpy(np.sort(idx)).to(flat.device)
    running = [b.reshape(-1) for n, b in net.named_buffers() if ".running_" in n and not n.startswith("FDS.")]
    arrays = {"loss": loss, "outputs": outputs, "encoding": encoding, "bn_running_stats": torch.cat(running),
              "parameters_sample": flat[idx], "gradients_sample": net.flat_grads()[idx]}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.detach().float().cpu().numpy())


def timed(fn, steps, warmup, world, device):
    import torch.distributed as dist
    for i in range(warmup):
        fn(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    for i in range(steps):
        fn(warmup + i)
    ev1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - t0
    dev_ms = ev0.elapsed_time(ev1)
    ms = torch.tensor([max(dev_ms, 0.0), wall * 1e3], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms[0]), float(ms[1])


def _bcast0(t):
    import torch.distributed as dist
    r = t.clone()
    dist.broadcast(r, 0)
    return r


def conv_flops_per_image():
    """Exact fprop / dgrad / wgrad FLOPs of the ResNet-50 conv stack per 224^2 image (2*M*N*K per GEMM)."""
    f = d = w = 0.0
    def conv(h, cin, cout, k, s, first=False):
        nonlocal f, d, w
        ho = (h + 2 * (k // 2) - k) // s + 1
        fl = 2.0 * ho * ho * cout * cin * k * k
        f += fl
        w += fl
        if not first:
            d += fl
        return ho
    h = conv(224, 3, 64, 7, 2, first=True)
    h = (h - 1) // 2 + 1
    inpl = 64
    for li, nb in enumerate((3, 4, 6, 3)):
        pl = 64 << li
        for b in range(nb):
            s = 2 if (b == 0 and li > 0) else 1
            conv(h, inpl, pl, 1, 1)
            h2 = conv(h, pl, pl, 3, s)
            conv(h2, pl, pl * 4, 1, 1)
            if b == 0:
                conv(h, inpl, pl * 4, 1, s)
            inpl, h = pl * 4, h2
    return f, d, w


def fds_roofline(device, peaks):
    """Achieved HBM GB/s of the FDS segmented accumulation at the two epoch sizes; algorithmic bytes = 4*N*D + 4*N
    (features read once + bins), L2 flushed between iterations.  Two timings per size, both CUDA events on the
    launching stream: `kernel_ms` = fds_accumulate_kernel alone (events recorded inside the C-ABI call,
    dirb200_fds_set_profiling) -> achieved_gbs / frac (the roofline figure of the dominant kernel); `call_ms` = the
    whole dirb200_fds_accumulate call (counting sort of the rows + the kernel) -> call_gbs / call_frac."""
    import ctypes
    import _lib
    d, nb = 2048, BUCKET_NUM - BUCKET_START
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    out = {}
    _lib.call("dirb200_fds_set_profiling", 1)
    for n in (256, 12208, 191509):
        feats = torch.relu(torch.randn(n, d, device=device) + 0.5)
        labels = torch.from_numpy(synthetic_labels(n, 3)).to(device)
        bins = labels.clamp(max=nb - 1).to(torch.int32)
        sums = torch.zeros(nb, d, dtype=torch.float64, device=device)
        sumsq = torch.zeros_like(sums)
        counts = torch.zeros(nb, dtype=torch.int64, device=device)
        need = int(_lib.raw("dirb200_fds_accumulate_workspace_bytes")(n, nb))
        ws = torch.empty(need, dtype=torch.uint8, device=device)
        st = _lib.stream_ptr()
        times, ktimes = [], []
        for it in range(8):
            flush.fill_(it)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.call("dirb200_fds_accumulate", _lib.ptr(feats), _lib.ptr(bins), n, d, nb, _lib.ptr(sums),
                      _lib.ptr(sumsq), _lib.ptr(counts), _lib.ptr(ws), need, st)
            e1.record()
            torch.cuda.synchronize()
            kms = ctypes.c_float(0.0)
            _lib.call("dirb200_fds_last_accumulate_kernel_ms", ctypes.byref(kms))
            if it >= 3:
                times.append(e0.elapsed_time(e1))
                ktimes.append(float(kms.value))
        ms, kms = float(np.mean(times)), float(np.mean(ktimes))
        alg = 4.0 * n * d + 4.0 * n
        out[str(n)] = {"kernel_ms": kms, "achieved_gbs": alg / kms / 1e6, "frac": alg / kms / 1e6 / peaks["hbm_gbs"],
                       "call_ms": ms, "call_gbs": alg / ms / 1e6, "call_frac": alg / ms / 1e6 / peaks["hbm_gbs"],
                       "algorithmic_mb": alg / 1e6}
        del feats, ws
    _lib.call("dirb200_fds_set_profiling", 0)
    # FDS.smooth (the fused whiten-recolor calibration, fwd) on one batch of 256: 2*B*D*4 bytes of features + the
    # rows of the four tables it touches; latency-bound at this size, reported in microseconds
    from fds import FDS
    m = FDS(d, BUCKET_NUM, BUCKET_START, kernel="gaussian", ks=5, sigma=2).to(device)
    for k in ("running_var_last_epoch", "smoothed_var_last_epoch"):
        getattr(m, k).uniform_(0.5, 1.5)
    x = torch.relu(torch.randn(256, d, device=device) + 0.5)
    lab = torch.from_numpy(synthetic_labels(256, 5)).to(device).reshape(-1, 1)
    ts = []
    for it in range(8):
        flush.fill_(it)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        m.smooth(x, lab, 2)
        e1.record()
        torch.cuda.synchronize()
        if it >= 3:
            ts.append(e0.elapsed_time(e1))
    alg = 2.0 * 256 * d * 4 + 256 * 4 + 4.0 * nb * d * 4
    out["calibrate_b256"] = {"call_us": 1e3 * float(np.mean(ts)), "algorithmic_mb": alg / 1e6,
                             "call_gbs": alg / float(np.mean(ts)) / 1e6,
                             "note": "FDS.smooth forward through the Python mirror (bin rows + fused calibrate kernel)"}
    return out


def run_ours(args):
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    json_fd = 1
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        # stdout must stay the one JSON line, but NCCL writes its banner ("NCCL version ...") and, at higher
        # NCCL_DEBUG levels, its whole log to file descriptor 1: keep a private copy of the real stdout for the JSON
        # line and point fd 1 at stderr for everything else this process (and the libraries in it) prints
        sys.stdout.flush()
        json_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=device)
    import _lib
    peaks = measured_peaks()
    model, opt, ep_labels, w_all = build_training_state(args, device, rank, world)

    # ---- (1) device-resident throughput: `value`
    dev_batches = make_batches(args, device, rank, ep_labels, w_all, pinned=False)
    last = [None]
    def step_resident(i):
        x, t, w = dev_batches[i % len(dev_batches)]
        last[0] = train_step(model, opt, x, t, w)
    sampler = ClockSampler(local)
    timed(step_resident, 0, args.warmup, world, device)
    launches0 = _lib.launch_count()
    sampler.start()
    dev_ms, wall_ms = timed(step_resident, args.steps, 0, world, device)
    clocks = sampler.stop()
    launches = _lib.launch_count() - launches0
    if args.dump_outputs and rank == 0:     # before the steps below change the model
        dump_outputs(args.dump_outputs, *last[0], model.module)
    last[0] = None
    ms_per_step = dev_ms / args.steps
    value = world * args.batch * args.steps / (dev_ms / 1e3)

    # ---- (2) end to end: pinned host batches, H2D every step (prefetched on a side stream), loss read back
    host_batches = make_batches(args, device, rank, ep_labels, w_all, pinned=True)
    copy_stream = torch.cuda.Stream()
    slots = [None, None]
    loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
    loss_events = [None, None]

    def prefetch(i):
        hb = host_batches[i % len(host_batches)]
        with torch.cuda.stream(copy_stream):
            slots[i % 2] = (tuple(a.to(device, non_blocking=True) for a in hb), copy_stream.record_event())

    def step_e2e(i):
        if slots[i % 2] is None:
            prefetch(i)
        (x, t, w), ev = slots[i % 2]
        torch.cuda.current_stream().wait_event(ev)
        prefetch(i + 1)
        loss = train_step(model, opt, x, t, w)[0]
        for a in (x, t, w):
            a.record_stream(torch.cuda.current_stream())
        if loss_events[i % 2] is not None:
            loss_events[i % 2].synchronize()          # the read of step i-2 has landed on the host
        loss_host[i % 2:i % 2 + 1].copy_(loss.detach().reshape(1), non_blocking=True)
        loss_events[i % 2] = torch.cuda.current_stream().record_event()

    e2e_dev_ms, e2e_wall_ms = timed(step_e2e, args.steps, max(3, args.warmup // 2), world, device)
    e2e_value = world * args.batch * args.steps / (max(e2e_dev_ms, e2e_wall_ms) / 1e3)
    h2d = sum(a.numel() * a.element_size() for a in host_batches[0])

    # ---- (3) per-kernel-class timing (profiling steps are NOT part of the numbers above)
    shape = (args.batch, 3, 224, 224)
    model.module.set_profiling(shape, True)
    for i in range(2):
        step_resident(i)
    prof = model.module.read_profile(shape)
    model.module.set_profiling(shape, False)
    prof = {k: (ms / 2, cnt // 2) for k, (ms, cnt) in prof.items()}
    f, d, wg = conv_flops_per_image()
    conv_ms = prof["conv_fprop"][0] + prof["conv_dgrad"][0] + prof["conv_wgrad"][0]
    conv_flops = (f + d + wg) * args.batch
    # DRAM traffic of the same kernels from the committed ncu launch list (profiles/r2_launches.json: sum of
    # dram__bytes_read + dram__bytes_write over the conv launches of one step), else null
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r2_launches.json")
    if os.path.exists(tpath) and args.batch == 256:
        traffic = json.load(open(tpath)).get("conv_dram_gb")
    nlaunch = prof['conv_fprop'][1] + prof['conv_dgrad'][1] + prof['conv_wgrad'][1]
    roofline = {"bound": "tensor", "kernel": "igemm_kernel (tcgen05 implicit-GEMM conv: fprop+dgrad+wgrad, "
                f"{nlaunch} launch groups/step; achieved = their summed algorithmic FLOPs / summed CUDA-event time)",
                "achieved": conv_flops / (conv_ms / 1e3) / 1e12, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                "frac": conv_flops / (conv_ms / 1e3) / 1e12 / peaks["bf16_sustained"], "traffic": traffic,
                "traffic_unit": "GB of DRAM read+write per step over these launches (ncu)",
                "peak_source": peaks["source"] + ", sustained (kernel timed inside a long step)",
                "algorithmic_gflop_per_step": conv_flops / 1e9, "kernel_ms_per_step": conv_ms,
                "note": "the timed launches also do BatchNorm work in their epilogues (fprop: batch statistics of its "
                        "output; 29 of the dgrads: the BN-backward moments of the previous layer, reading y once more) -- "
                        "that time is counted here, the FLOPs are the convolutions' only"}
    breakdown = {k: {"ms_per_step": round(ms, 4), "launch_groups": cnt} for k, (ms, cnt) in prof.items()}

    # ---- (4) multi-GPU correctness evidence: after the timed steps every replica must hold bit-identical parameters
    # and FDS tables (same all-reduced gradients, same all-reduced statistics): max |p_rank - p_0| over the ranks
    replica_check = None
    if world > 1:
        flat = model.module.flat_parameters()
        ref = flat.clone()
        dist.broadcast(ref, 0)
        diffs = torch.stack([(flat - ref).abs().max(),
                             (model.module.FDS.running_mean - _bcast0(model.module.FDS.running_mean)).abs().max(),
                             (model.module.FDS.smoothed_var_last_epoch
                              - _bcast0(model.module.FDS.smoothed_var_last_epoch)).abs().max()]).double()
        dist.all_reduce(diffs, op=dist.ReduceOp.MAX)
        replica_check = {"max_abs_param_diff_vs_rank0": float(diffs[0]), "max_abs_fds_running_mean_diff": float(diffs[1]),
                         "max_abs_fds_smoothed_var_diff": float(diffs[2]), "param_l1": float(flat.double().abs().sum())}

    out = None
    if rank == 0:
        fds_rf = fds_roofline(device, peaks)
        cpu = cpu_baseline_sample() if (world == 1 and not args.no_cpu_baseline) else None
        out = {"metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
               "config": {"workload": WORKLOAD, "batch_per_gpu": args.batch, "global_batch": args.batch * world,
                          "parallelism": f"dp{world}", "l2": "per-step working set (~11 GB of activations) >> 126 MB L2; "
                          f"{args.num_batches} distinct input batches", "timing": "CUDA events, max over ranks"},
               "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                       "ms_per_step": max(e2e_dev_ms, e2e_wall_ms) / args.steps},
               "roofline": roofline, "fds_roofline": {"bound": "hbm", "kernel": "fds_accumulate_kernel (achieved/frac: the "
                                                      "kernel alone; call_*: whole dirb200_fds_accumulate incl. the "
                                                      "counting sort)", "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                                      "peak_source": peaks["source"] + ", burst (kernel timed alone)",
                                                      "by_rows": fds_rf},
               "cpu_baseline": cpu, "clocks": clocks, "gpu_launches": int(launches),
               "gpu_launches_per_step": launches / args.steps, "wall_ms_per_step": wall_ms / args.steps,
               "kernel_breakdown_ms": breakdown,
               "kernel_breakdown_note": "from 2 extra profiling-mode steps (CUDA events around every launch group: "
                                        "their sum exceeds ms_per_step by the event overhead); not part of the timed steps",
               "model_flops_utilisation": FWDBWD_GFLOP_PER_IMG * args.batch / ms_per_step / SPEC_BF16_TFLOPS,
               "model_flops_utilisation_note": "24.29 GFLOP/img fwd+bwd vs the nominal dense bf16 peak (2250 TFLOP/s)",
               "step_frac_of_measured_bf16_peak": FWDBWD_GFLOP_PER_IMG * args.batch / ms_per_step / peaks["bf16_sustained"],
               "replica_check": replica_check}
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--num-batches", dest="num_batches", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-batch", dest="cpu_batch", type=int, default=16,
                    help="images per step of the CPU arm (a bounded sample of the 256-image step)")
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU arm's outputs (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
