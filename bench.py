#!/usr/bin/env python
"""bench.py — query images/sec of the OnePose++ 2D-3D matcher hot path on B200.

    python bench.py --gpus 1 --steps 20 --warmup 3            # our CUDA path, one JSON line
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   # N > 1
    python bench.py --impl reference --steps K --warmup W      # reference CPU arm (oracle port)

A "step" is one forward of ``OnePosePlus_model`` over a batch of 512x512 query images against a
5000-point planted descriptor bank (BASELINE.json configs[2]: batch 64 on one GPU; with N GPUs the
image batch is sharded 64 per GPU = configs[3], weak scaling; the bank is NCCL-broadcast once).
``value`` is whole-job images/s with inputs resident in HBM; ``e2e`` is the same metric through
the public ``model(data)`` call with pinned-host inputs (H2D) and match results read back (D2H)
inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = W = 512
N_POINTS = 5000
N_PLANTED = 3000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="images per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-ops", action="store_true", help="print the per-op breakdown to stderr")
    ap.add_argument("--no-c5", action="store_true", help="skip the BASELINE configs[4] block")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (see dump_outputs)")
    return ap.parse_args()


DUMP_BUDGET = 64 << 20     # bytes written by --dump-outputs, at most
DUMP_SEED = 0


def dump_outputs(out_dir, data, input_keys):
    """Write what one forward returned to its caller (every key of `data` not in `input_keys`) as
    out_dir/<name>.npy: float tensors in float32 (float64 stays float64), integer and bool tensors
    and Python scalars / shapes in float64 (exact).  A tensor of more than 2**20 entries is written
    as a fixed sample of 2**20 of its flattened entries (seeded by DUMP_SEED, ascending flat indices
    in <name>_sample_index.npy), halved until all files fit in DUMP_BUDGET.
    With the same bench arguments the inputs are the same, so the files of two builds compare
    entry for entry."""
    arrays = {}
    for k, v in data.items():
        if k in input_keys or v is None:
            continue
        t = v.detach() if torch.is_tensor(v) else torch.tensor(v, dtype=torch.float64)
        if t.is_floating_point() and t.dtype != torch.float64:
            t = t.float()
        elif not t.is_floating_point():
            t = t.double()
        arrays[k] = t

    def nbytes(cap):
        return sum(min(t.numel(), cap) * t.element_size() + (8 * cap if t.numel() > cap else 0)
                   for t in arrays.values())
    cap = 1 << 20
    while nbytes(cap) > DUMP_BUDGET:
        cap //= 2
    os.makedirs(out_dir, exist_ok=True)
    for k, t in arrays.items():
        if t.numel() > cap:
            g = torch.Generator().manual_seed(DUMP_SEED)
            idx = torch.randint(0, t.numel(), (cap,), generator=g).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
            np.save(os.path.join(out_dir, k + "_sample_index.npy"), idx.double().numpy())
        np.save(os.path.join(out_dir, k + ".npy"), t.cpu().numpy())


# ---------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md: sample nvidia-smi DURING the timed region)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons of the GPU while the timed region runs (B200_PROFILING.md's clocks
    line).  Read through NVML in this process (the counters nvidia-smi prints; a poll costs tens of
    microseconds) — a looping `nvidia-smi -lms 100` child was seen to slow the eager-mode timed region
    it overlapped by 5-8 % on some boxes (driver lock held during its queries) while the later,
    unsampled regions of the same run were not affected.  Falls back to `nvidia-smi -lms 200`."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
            ("sw_power_cap", 0x4))     # nvmlClocksEventReason* masks

    def __init__(self, index):
        self.rows = []      # (time, sm_mhz, max_mhz, set(reasons))
        self.proc = None
        self.source = None
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                ent = vis.split(",")[index].strip()
                phys = int(ent) if ent.isdigit() else None
            h = pynvml.nvmlDeviceGetHandleByIndex(phys) if phys is not None else pynvml.nvmlDeviceGetHandleByUUID(ent)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def poll():
                while not self._stop.is_set():
                    try:
                        sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        mask = int(reasons_fn(h))
                        self.rows.append((time.time(), sm, mx, {n for n, b in self.BITS if mask & b}))
                    except Exception:  # noqa: BLE001
                        pass
                    self._stop.wait(0.25)
            poll_once_ok = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)) > 0
            if poll_once_ok:
                self.source = "nvml"
                self.t = threading.Thread(target=poll, daemon=True)
                self.t.start()
                return
        except Exception:  # noqa: BLE001  (no NVML: use the CLI)
            pass
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi -lms 200"
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            try:
                sm, mx = float(f[0]), float(f[1])
            except (ValueError, IndexError):
                continue
            names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
            self.rows.append((time.time(), sm, mx, {n for n, v in zip(names, f[2:6]) if v == "Active"}))

    def stop(self, t0, t1):
        if self.source is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi / NVML unavailable"]}
        self._stop.set()
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, s_mhz, m_mhz, rs in list(self.rows):
            if ts < t0 or ts > t1:
                continue
            sm.append(s_mhz)
            mx = m_mhz
            reasons |= rs
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm), "source": self.source}


# ---------------------------------------------------------------------------------------------
# reference arm: the CPU implementation of the path on the host cores (oracle port)
# ---------------------------------------------------------------------------------------------
def best_cpu_threads(fn):
    """The oracle is torch-CPU: try a few intra-op thread counts (a cgroup-limited box reports more
    cores than it can run) and keep the fastest, so the CPU baseline is its best, not an
    oversubscribed run."""
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cands = sorted({c for c in (8, 16, 32, 64, torch.get_num_threads(), ncpu) if 1 <= c <= ncpu})
    best, best_t = cands[0], float("inf")
    fn()
    for c in cands:
        torch.set_num_threads(c)
        t = time.perf_counter()
        fn()
        dt = time.perf_counter() - t
        if dt < best_t:
            best, best_t = c, dt
        if dt > 4 * best_t:
            break
    torch.set_num_threads(best)
    return best


def run_reference(args, rank):
    if rank != 0:
        return
    from oracle import oracle, workload
    sd = workload.synthetic_state_dict(0)
    data, _ = workload.planted_workload(sd, H, W, N_POINTS, N_PLANTED, batch=1)
    cores = best_cpu_threads(lambda: oracle.forward(sd, {k: v.clone() for k, v in data.items()}))
    sample = 1  # images per step: bounded sample of the batch-64 workload

    def step():
        d = {k: v.clone() for k, v in data.items()}
        oracle.forward(sd, d)
        return d

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        d = step()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, d, set(data))
    val = sample * args.steps / dt
    print(json.dumps({
        "impl": "reference", "metric": "query images/sec (512x512, 5k 3D pts)", "value": val,
        "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (planted descriptors, seeded weights)",
        "config": {"workload": "BASELINE configs[2] shape (512x512 images, 5000-pt bank); each step is "
                               "a bounded sample of 1 image of the batch", "matches_per_image": int(d["b_ids"].numel())},
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} forwards of 1 image (oracle/oracle.py, torch CPU fp32)"},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def conv_flops_table(B, h=H, w=W, head=True):
    """Algorithmic MACs of the tcgen05 conv launches of one backbone pass (true channel counts;
    the 7x7 conv1 — 0.41 GMAC/image — is listed separately).  head=False: without
    layer1_outconv2, which the forward evaluates on the match windows only."""
    h2, h4, h8 = (h // 2) * (w // 2), (h // 4) * (w // 4), (h // 8) * (w // 8)
    macs = 0
    macs += 4 * h2 * 128 * 128 * 9                                   # layer1
    macs += h4 * 196 * 128 * 9 + 3 * h4 * 196 * 196 * 9 + h4 * 196 * 128   # layer2 (+downsample)
    macs += h8 * 256 * 196 * 9 + 3 * h8 * 256 * 256 * 9 + h8 * 256 * 196   # layer3
    macs += h8 * 256 * 256 + h4 * 256 * 196 + h4 * 256 * 256 * 9 + h4 * 196 * 256 * 9   # fpn 1/4
    macs += h2 * 196 * 128                                                             # fpn 1/2 lateral
    if head:
        macs += h2 * 196 * 196 * 9 + h2 * 128 * 196 * 9                                # layer1_outconv2
    return 2.0 * macs * B


def ncu_traffic(kernel_substr, launch_index):
    """DRAM bytes (read + write) of one launch from the committed ncu capture at the bench batch
    (profiles/r2_ncu_b64_raw.csv: kernel name, launch index, dram__bytes_read.sum, dram__bytes_write.sum),
    or None when no capture at this batch is committed — never a scaled constant."""
    path = os.path.join(ROOT, "profiles", "r2_ncu_b64_traffic.json")
    try:
        t = json.load(open(path))
        e = t[kernel_substr][launch_index]
        return e["dram_read_bytes"] + e["dram_write_bytes"]
    except (OSError, KeyError, IndexError, ValueError):
        return None


def cuda_time(fn, reps, warm=2):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def bench_c5(model, sd, dev, workload, peaks, steps=5, batch=8):
    """BASELINE configs[4]: 640x480 images (60x80 = 4800 coarse cells) vs a 20 000-point bank, fine
    window 5 — the configuration whose (H/8*W/8) x N score matrix stresses HBM: conf_matrix is
    384 MB per image.  Reports images/s with the matrix materialised (reference contract) and
    without (lazy), and the dual-softmax passes alone against the measured HBM peak."""
    h, w, n = 480, 640, 20000
    data, _ = workload.planted_workload(sd, h, w, n, 6000, batch=1)
    g = torch.Generator().manual_seed(5)
    imgs = (data["query_image"] + 0.02 * torch.randn(batch, 1, h, w, generator=g)).clamp(0, 1).to(dev)
    scale = data["query_image_scale"].expand(batch, -1).contiguous().to(dev)
    bank = {k: data[k].to(dev) for k in ("keypoints3d", "descriptors3d_db", "descriptors3d_coarse_db")}
    out = {}

    def step():
        d = {"query_image": imgs, "query_image_scale": scale, **bank}
        model(d)
        out["d"] = d

    res = {"workload": f"BASELINE configs[4]: batch {batch} images 640x480 vs shared 20000-pt bank, window 5",
           "conf_matrix_bytes_per_image": 4 * n * (h // 8) * (w // 8)}
    for mode in ("eager", "lazy"):
        model.conf_matrix_mode = mode
        ms = cuda_time(step, steps)
        res[f"images_per_s_conf_{mode}"] = batch / ms * 1e3
        res[f"ms_per_step_conf_{mode}"] = ms
    res["matches_per_image"] = out["d"]["b_ids"].numel() / batch
    # the dual-softmax passes alone (coarse_matching.py:102-119) on the final tokens of the last step
    S = (h // 8) * (w // 8)
    pl = 2 if model.split else 1
    q2 = model._buf("q2_0", (batch, S, pl * 256), torch.float16, dev)
    d3 = model._buf("d3_0", (batch, n, pl * 256), torch.float16, dev)
    bstate = {"Bb": 1, "N": n, "kpts": bank["keypoints3d"].float().contiguous()}
    for mode in ("eager", "lazy"):
        model.conf_matrix_mode = mode
        ms = cuda_time(lambda: model._coarse_matching(q2, d3, bstate, scale, batch, n, h // 8, w // 8, 8.0, {}), steps)
        alg = batch * (n + S) * pl * 256 * 2 * 2 + (batch * n * S * 4 if mode == "eager" else 0)
        res[f"sim_passes_ms_conf_{mode}"] = ms
        res[f"sim_passes_hbm_gbs_conf_{mode}"] = alg / ms / 1e6
        res[f"sim_passes_hbm_frac_conf_{mode}"] = alg / ms / 1e6 / peaks.get("hbm_gbs", 6562.6)
    res["note"] = ("sim-pass bytes = tokens read once per GEMM pass (2 passes) + the fp32 conf_matrix store when "
                   "materialised; 2*2*20000*4800*256 flop per image and pass on the tensor pipe (x3 issued)")
    model.conf_matrix_mode = "eager"
    return res


def bench_loftr(dev, workload, steps=5, batch=8):
    """SURVEY §8 f3: the 2D-2D matcher (LoFTR_for_OnePose_Plus) on the same engine — image pairs/s at
    batch 8 of 512x512 pairs (= 16 backbone images, 8 coarse layers on 2 x 4096 tokens, 9x9 fine
    windows), planted pair so that hundreds of matches reach the fine level."""
    from onepose_plus_plus_b200 import LoFTR_for_OnePose_Plus
    from oracle import loftr_oracle
    sd, data = workload.planted_loftr(512, 512, batch=1)
    m = LoFTR_for_OnePose_Plus(loftr_oracle.DEFAULT_CONFIG)
    m.load_state_dict(sd, strict=True)
    m = m.eval().to(dev)
    g = torch.Generator().manual_seed(9)
    im0 = (data["image0"] + 0.005 * torch.randn(batch, 1, 512, 512, generator=g)).clamp(0, 1).to(dev)
    im1 = (data["image1"] + 0.005 * torch.randn(batch, 1, 512, 512, generator=g)).clamp(0, 1).to(dev)
    out = {}

    def step():
        d = {"image0": im0, "image1": im1}
        m(d)
        out["d"] = d

    ms = cuda_time(step, steps)
    return {"workload": f"batch {batch} pairs of 512x512 images, fine window 9 (loftr_for_onepose_plus_cfg.py)",
            "pairs_per_s": batch / ms * 1e3, "ms_per_step": ms,
            "matches_per_pair": out["d"]["b_ids"].numel() / batch}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch.distributed as dist
    from onepose_plus_plus_b200 import OnePosePlus_model, _lib, ops, parallel
    from oracle import oracle, workload  # checkpoint + workload generators and the cpu_baseline leg only

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # started now so that nvidia-smi is already streaming when the (short) timed region begins
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_burst = peaks.get("bf16_tflops", 1590.0)   # for a kernel timed alone (B200_PROFILING.md)
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback"

    B = args.batch
    sd = workload.synthetic_state_dict(0)
    model = OnePosePlus_model(oracle.DEFAULT_CONFIG)
    model.load_state_dict(sd, strict=True)
    model = model.eval().to(dev)

    # per-object descriptor bank: built on rank 0, NCCL-broadcast once (SURVEY §8e); every rank
    # derives its own image shard from the same base image (seeded per rank)
    data, _ = workload.planted_workload(sd, H, W, N_POINTS, N_PLANTED, batch=1)
    bank = {k: data[k].to(dev) for k in ("keypoints3d", "descriptors3d_db", "descriptors3d_coarse_db")}
    if world > 1:
        for k in bank:
            if rank != 0:
                bank[k].zero_()          # prove the bank really arrives over NCCL
        parallel.broadcast_bank(bank, src=0)
    g = torch.Generator().manual_seed(100 + rank)
    base = data["query_image"]
    imgs_f = (base + 0.02 * torch.randn(B, 1, H, W, generator=g)).clamp(0, 1)
    imgs8_host = (imgs_f * 255).round().to(torch.uint8).pin_memory()          # what a camera / decoder delivers
    imgs_host = (imgs8_host.float() / 255).pin_memory()                       # data_io.py:107 (reference input)
    scale_host = data["query_image_scale"].expand(B, -1).contiguous().pin_memory()
    bank_host = {k: v.cpu().pin_memory() for k, v in bank.items()}

    def make_data(images, scale, bk):
        # the reference's data dict: the bank rides along with every call (one object, [1, N, .])
        return {"query_image": images, "query_image_scale": scale, **bk}

    imgs_dev = imgs_host.to(dev)
    scale_dev = scale_host.to(dev)

    def step_resident():
        d = make_data(imgs_dev, scale_dev, bank)
        model(d)
        return d

    out_host = {}
    lo = rank * B

    def read_back(d):
        if world > 1:    # the one data-plane collective: every rank's matches to every rank
            out_host["all"] = parallel.gather_matches(d, lo).cpu()
        else:
            for k in ("mkpts_3d_db", "mkpts_query_f", "mconf", "m_bids"):
                out_host[k] = d[k].cpu()

    def step_e2e_refapi():
        # the reference worker's loop (inference_OnePosePlus_worker.py:54-56): fp32 frames AND the bank
        # go host -> device with every call
        im = imgs_host.to(dev, non_blocking=True)
        sc = scale_host.to(dev, non_blocking=True)
        bk = {k: v.to(dev, non_blocking=True) for k, v in bank_host.items()}
        d = make_data(im, sc, bk)
        model(d)
        read_back(d)
        return d

    def step_e2e():
        # this repo's input path: bank resident (set_bank, once per object), uint8 frames
        im = imgs8_host.to(dev, non_blocking=True)
        sc = scale_host.to(dev, non_blocking=True)
        d = {"query_image": im, "query_image_scale": sc}
        model(d)
        read_back(d)
        return d

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_ms = []

    def timed(fn, steps, per_step=False):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = []
        t0 = time.time()
        e0.record()
        for _ in range(steps):
            d = fn()
            if per_step:       # diagnostics only: an event record costs nothing on the stream
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                marks.append(ev)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if per_step:
            prev = e0
            for ev in marks:
                step_ms.append(round(prev.elapsed_time(ev), 3))
                prev = ev
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), d, t0, time.time()

    # untimed settle phase (allocator high-water marks, power state: the first timed region of a fresh
    # process was seen 8 % slower than the later ones of the same run on some boxes — the power-cap
    # controller needs a second or two of the real load), then the W >= 3 warm-up steps of the contract
    t_settle, n_settle = time.time(), 0
    while n_settle < 5 or time.time() - t_settle < 2.5:     # >= 5 steps and >= 2.5 s under load
        d = step_resident()
        torch.cuda.synchronize()
        n_settle += 1
    for _ in range(max(args.warmup, 3)):
        d = step_resident()
    _lib.LAUNCHES = 0
    ms, d, t0, t1 = timed(step_resident, args.steps, per_step=True)
    clocks = sampler.stop(t0, t1) if sampler else None
    if args.dump_outputs and rank == 0:     # before any later forward reuses the workspace
        dump_outputs(args.dump_outputs, d, set(make_data(imgs_dev, scale_dev, bank)))
    launches = _lib.LAUNCHES
    m_per_img = d["b_ids"].numel() / B

    # same step without materialising conf_matrix (no inference consumer reads it)
    model.conf_matrix_mode = "lazy"
    for _ in range(2):
        step_resident()
    ms_lazy, _, _, _ = timed(step_resident, args.steps)
    model.conf_matrix_mode = "eager"

    for _ in range(2):
        step_e2e_refapi()
    ms_e2e_ref, _, _, _ = timed(step_e2e_refapi, args.steps)
    h2d_ref = imgs_host.numel() * 4 + scale_host.numel() * 4 + sum(v.numel() * 4 for v in bank_host.values())
    model.set_bank(bank["keypoints3d"], bank["descriptors3d_db"], bank["descriptors3d_coarse_db"])
    for _ in range(2):
        step_e2e()
    ms_e2e, d2, _, _ = timed(step_e2e, args.steps)
    model.clear_bank()
    h2d = imgs8_host.numel() + scale_host.numel() * 4
    d2h = sum(v.numel() * v.element_size() for v in out_host.values())

    # pose stage on the device (SURVEY §8 f1): matcher + batched RANSAC-PnP per step, vs the
    # reference's per-frame cv2.solvePnPRansac on the host (metric_utils.py:121-204)
    pose = None
    if rank == 0:
        try:
            from onepose_plus_plus_b200 import pnp as dpnp
            Kmat = torch.tensor([[600.0, 0, W / 2], [0, 600.0, H / 2], [0, 0, 1]], device=dev).expand(B, 3, 3).contiguous()

            def step_pose():
                dd = step_resident()
                return dd, dpnp.ransac_pnp_batched(dd["m_bids"], dd["mkpts_3d_db"], dd["mkpts_query_f"], Kmat,
                                                   reprojection_error=5.0)
            ms_pose = cuda_time(lambda: step_pose(), max(args.steps // 2, 3))
            dd, rr = step_pose()
            ms_pnp = cuda_time(lambda: dpnp.ransac_pnp_batched(dd["m_bids"], dd["mkpts_3d_db"], dd["mkpts_query_f"],
                                                               Kmat, reprojection_error=5.0), 5)
            pose = {"frames_per_s_matcher_plus_pnp": B / ms_pose * 1e3, "ms_per_step": ms_pose,
                    "pnp_ms_per_batch": ms_pnp, "pnp_us_per_frame": ms_pnp / B * 1e3,
                    "matches_per_frame": dd["m_bids"].numel() / B,
                    "note": "opp_pnp_ransac: one CTA per frame, 1024 P3P hypotheses + 3 Gauss-Newton refinement "
                            "rounds, consuming the match lists in place (no D2H before the pose)"}
            if world == 1 and not args.no_cpu_baseline:
                from oracle import pnp as opnp      # cpu_baseline leg: the reference's cv2 call, one frame
                sel = dd["m_bids"] == 0
                p2 = dd["mkpts_query_f"][sel].cpu().numpy()
                p3 = dd["mkpts_3d_db"][sel].cpu().numpy()
                t_c = time.perf_counter()
                for _ in range(5):
                    opnp.ransac_pnp(Kmat[0].cpu().numpy(), p2, p3, pnp_reprojection_error=5)
                pose["cpu_cv2_ms_per_frame"] = (time.perf_counter() - t_c) / 5 * 1e3
        except Exception as e:  # noqa: BLE001
            pose = {"error": f"{type(e).__name__}: {str(e)[:300]}"}

    # BASELINE configs[1] (one image per forward): latency view of the same path, wall clock incl.
    # host launch overhead and the per-forward match-count sync
    b1 = None
    if rank == 0:
        try:
            d1 = {"query_image": imgs_dev[:1].contiguous(), "query_image_scale": scale_dev[:1].contiguous(), **bank}
            for _ in range(3):
                model(dict(d1))
            torch.cuda.synchronize()
            n1, t_b1 = 20, time.perf_counter()
            for _ in range(n1):
                o1 = dict(d1)
                model(o1)
            torch.cuda.synchronize()
            dt1 = (time.perf_counter() - t_b1) / n1
            b1 = {"workload": "BASELINE configs[1]: one 512x512 image vs the 5000-pt bank (batch 1)",
                  "ms_per_image_eager": dt1 * 1e3, "matches": int(o1["b_ids"].numel()),
                  "timing": f"wall clock over {n1} back-to-back forwards (host launches + match-count sync included)"}
            # latency mode: resident bank, CUDA-graph replay, conf_matrix on demand
            model.set_bank(bank["keypoints3d"], bank["descriptors3d_db"], bank["descriptors3d_coarse_db"])
            model.enable_cuda_graphs(True)
            model.conf_matrix_mode = "lazy"
            dg = {"query_image": imgs_dev[:1].contiguous(), "query_image_scale": scale_dev[:1].contiguous()}
            for _ in range(3):
                model(dict(dg))
            torch.cuda.synchronize()
            t_b1 = time.perf_counter()
            for _ in range(n1):
                og = dict(dg)
                model(og)
            torch.cuda.synchronize()
            dtg = (time.perf_counter() - t_b1) / n1
            model.enable_cuda_graphs(False)
            model.conf_matrix_mode = "eager"
            model.clear_bank()
            b1.update({"ms_per_image": dtg * 1e3, "images_per_s": 1.0 / dtg,
                       "mode": "model.set_bank + enable_cuda_graphs() + conf_matrix_mode='lazy' (one graph launch, "
                               "one host sync at the end); ms_per_image_eager = the plain reference-API call",
                       "matches_graph": int(og["b_ids"].numel())})
        except Exception as e:  # noqa: BLE001  (auxiliary number: never lose the bench line over it)
            b1 = {"error": f"{type(e).__name__}: {str(e)[:200]}"}

    # dominant kernel: the tcgen05 implicit-GEMM conv engine (21 launches / forward), timed live
    # with CUDA events around the backbone on the launching stream
    conv_ms = attn_ms = l1_ms = None
    S_tok = (H // 8) * (W // 8)
    c5 = loftr = None
    if rank == 0:
        # the backbone as the forward runs it: everything up to layer1_outconv2, whose two 3x3
        # convolutions are evaluated afterwards on the 5x5 windows of the matches only
        conv_ms = cuda_time(lambda: model._backbone(imgs_dev, defer_fine=True), 3)
        x1_lat = model._backbone(imgs_dev, defer_fine=True)[1]
        head_dense_ms = cuda_time(lambda: model._fine_head_dense(x1_lat), 3)
        dm = {"query_image": imgs_dev, "query_image_scale": scale_dev, **bank}
        model(dm)
        x1_lat = model._backbone(imgs_dev, defer_fine=True)[1]
        Mh = int(dm["b_ids"].numel())
        head_win_ms = cuda_time(lambda: model._fine_head_windows(x1_lat, dm["b_ids"], dm["j_ids"], Mh,
                                                                 W // 8, 4), 3) if Mh else None
        fine_head = {"what": "layer1_outconv2 (3x3 208->208 + 3x3 208->128 at 1/2 resolution)",
                     "dense_ms": head_dense_ms, "windows_ms": head_win_ms, "matches": Mh,
                     "mode": model.fine_windows,
                     "note": "windows = the same convolutions on the 7x7 / 5x5 neighbourhood of each coarse match "
                             "(what fine_preprocess.py:40-47 reads); bit-equal outputs (tests)"}
        # the dominant kernel launch: layer1 3x3 conv 128->128 at 1/2 resolution (4 identical launches
        # per forward = 30 % of the conv flops), timed alone on the launching stream.  Its input
        # (batch x 256 x 256 x 2 planes x 128 ch fp16 = 2.1 GB at batch 64) exceeds L2.
        pl_ = 2 if model.split else 1
        x0 = model._buf("x0", (B, H // 2, W // 2, pl_ * 128), torch.float16, dev)
        y0 = model._buf("l1a_t", (B, H // 2, W // 2, pl_ * 128), torch.float16, dev)
        wl1, bl1 = model._plan["layer1.0.conv1"]
        l1_ms = cuda_time(lambda: ops.conv2d_nhwc(x0, wl1, bl1, y0, 3, 1, model.split, act=1), 5, warm=3)
        # coarse attention (BASELINE.json "coarse-attn tensor-pipe %"): the 6-layer linear-attention
        # transformer on both sequences (tcgen05 GEMM launches + the KV-state kernels), one object
        # per image so that nothing is served from the per-object cache
        q2, _, (hc, wc) = model._backbone(imgs_dev, defer_fine=True)
        S_tok = hc * wc
        bstate = {"Bb": B, "N": N_POINTS,
                  "d3_in": ops.to_planes(torch.randn(B, N_POINTS, 256, device=dev), model.split)}
        q2c = q2.clone()
        attn_ms = cuda_time(lambda: model._coarse_transformer(q2c, bstate, B, S_tok, N_POINTS), 3)
        if args.profile_ops:
            _lib.profile_ops(lambda: step_resident(), sys.stderr)
        if world == 1 and not args.no_c5:
            try:
                c5 = bench_c5(model, sd, dev, workload, peaks)
            except Exception as e:  # noqa: BLE001
                c5 = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
            try:
                model.clear_workspace()
                loftr = bench_loftr(dev, workload)
            except Exception as e:  # noqa: BLE001
                loftr = {"error": f"{type(e).__name__}: {str(e)[:300]}"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        d1, _ = workload.planted_workload(sd, H, W, N_POINTS, N_PLANTED, batch=1)
        best_cpu_threads(lambda: oracle.forward(sd, {k: v.clone() for k, v in d1.items()}))
        n_cpu = 8
        t = time.perf_counter()
        for _ in range(n_cpu):
            oracle.forward(sd, {k: v.clone() for k, v in d1.items()})
        dt = time.perf_counter() - t
        cpu = {"value": n_cpu / dt, "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"{n_cpu} forwards of 1 image of the same workload (oracle/oracle.py, torch CPU fp32)"}

    if rank == 0:
        total_imgs = B * world * args.steps
        flops = conv_flops_table(B, head=False)
        ach = flops / (conv_ms * 1e-3) / 1e12 if conv_ms else None
        passes = 3 if model.split else 1
        l1_flops = 2.0 * B * (H // 2) * (W // 2) * 128 * 128 * 9
        l1_tf = l1_flops / (l1_ms * 1e-3) / 1e12
        attn_flops = 2.0 * ((S_tok + N_POINTS) * 6 * 10 * 256 * 256 + (S_tok + N_POINTS) * 6 * 2 * 256 * 32) * B
        attn_tf = attn_flops / (attn_ms * 1e-3) / 1e12
        line = {
            "metric": "query images/sec (512x512, 5k 3D pts)",
            "value": total_imgs / (ms * 1e-3), "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp16 hi+lo operand pairs, 3 tcgen05 MMAs per K-step, fp32 accumulate (fp32-grade)"
                     if model.split else "f16",
            "data": "synthetic (seeded weights, planted descriptor bank, noisy copies of one image)",
            "config": {"workload": f"BASELINE configs[2]/[3]: batch {B} images 512x512 per GPU vs shared "
                                   f"5000-pt bank (NCCL-broadcast once when N>1)",
                       "global_batch": B * world, "matches_per_image": m_per_img,
                       "l2": "per-step working set (activations >= 1 GB) exceeds the 126 MB L2; no explicit flush",
                       "settle_steps": n_settle, "step_ms": step_ms,
                       "conf_matrix": "materialised fp32 every step (reference API); see conf_lazy for the "
                                      "store-free mode"},
            "clocks": clocks,
            "e2e": {"value": total_imgs / (ms_e2e * 1e-3), "unit": "images/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "model.set_bank(...) once per object, then model({'query_image': uint8 frames, "
                           "'query_image_scale': ...}) per step; pinned host buffers, match lists read back"
                           + ("; all-gather of every rank's matches (parallel.gather_matches) inside the timed region"
                              if world > 1 else "")},
            "e2e_reference_api": {"value": total_imgs / (ms_e2e_ref * 1e-3), "unit": "images/s",
                                  "h2d_bytes_per_step": h2d_ref, "d2h_bytes_per_step": d2h,
                                  "api": "the reference worker's call: fp32 frames + the whole bank uploaded with "
                                         "every model(data) (inference_OnePosePlus_worker.py:54-56)"},
            "conf_lazy": {"value": total_imgs / (ms_lazy * 1e-3), "unit": "images/s",
                          "ms_per_step": ms_lazy / args.steps,
                          "note": "model.conf_matrix_mode='lazy': data['conf_matrix'] is a handle that "
                                  "materialises on demand; matches identical (tests)"},
            "gpu_launches": launches,
            "roofline": {"bound": "tensor",
                         "kernel": "gemm_kernel<A_CONV,EpiConv>: layer1 3x3 conv 128->128 @256x256 (one launch, whole batch)",
                         "achieved": l1_tf, "peak": peak_burst, "unit": "TFLOP/s", "frac": l1_tf / peak_burst,
                         "traffic": ncu_traffic("EpiConv", 0),   # launch 0 = layer1.0.conv1, the launch timed here
                         "peak_source": peak_src.replace("bf16_tflops_sustained", "bf16_tflops (burst: kernel timed alone)"), "ms_per_launch": l1_ms,
                         "algorithmic_flops_per_launch": l1_flops, "mma_passes": passes,
                         "issued_tensor_tflops": l1_tf * passes, "issued_frac": l1_tf * passes / peak_burst,
                         "note": "achieved = algorithmic flops (2*B*256*256*128*128*9, reference fp32 math) / CUDA-event "
                                 "time of the launch; the fp32-grade mode issues mma_passes x that on the tensor pipe; "
                                 "traffic = dram read+write of this launch from the committed ncu --set full capture at "
                                 "this batch (profiles/r2_ncu_b64_traffic.json), null when absent",
                         "backbone": {"kernels": "conv1 im2col + 20 tcgen05 GEMM launches (FPN upsample-adds fused), without layer1_outconv2",
                                      "ms": conv_ms, "fine_head": fine_head,
                                      "algorithmic_tflops": ach, "frac": ach / peak_tf if ach else None,
                                      "issued_frac": ach * passes / peak_tf if ach else None}},
            "coarse_attention": {
                "kernels": "gemm_kernel<A_ROWS,{EpiStoreF16,EpiQ,EpiLN}> x60 + kv_partial/kv_finalize x12",
                "ms": attn_ms, "algorithmic_tflops": attn_tf, "issued_tensor_tflops": attn_tf * passes,
                "frac_of_peak_algorithmic": attn_tf / peak_tf, "frac_of_peak_issued": attn_tf * passes / peak_tf,
                "flops_per_image": "(4096 + 5000) tokens x 6 layers x 10*d^2 MAC + KV/QKV contractions = 72.6 GFLOP",
                "tensor_pipe_pct_ncu": "sm__pipe_tensor_cycles_active per launch at this batch: profiles/r2_ncu_xfmr_b64.md"},
            "configs": {"c5": c5, "loftr_2d2d": loftr},
            "pose_stage": pose,
            "latency_b1": b1,
            "kernel_options": {"lib": os.path.basename(_lib.LIB_PATH),
                               "one_pass_dual_softmax": bool(model.coarse_colmax and model.coarse_lse_cols),
                               "kv_single_plane": bool(model.kv_single_plane)},
            "cpu_baseline": cpu,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
