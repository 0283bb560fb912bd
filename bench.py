#!/usr/bin/env python
"""bench.py — BASELINE.json's metric: 3-stage 256x256 speech-conditioned StackGAN-v2 TRAIN images/sec.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch 24] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...   (N > 1)

One "step" = the reference's inner train loop over one batch (trainer.py:537-572 minus Inception): G forward,
3 x train_Dnet (real/wrong/fake passes, BCE, backward, Adam), train_Gnet (D forwards, BCE + class-aware + KL, backward
through Ds and G, Adam), EMA. Workload = BASELINE.json configs[1]: birds_3stages.yml, batch 24 per GPU, synthetic
inputs, random-init (weights_init) weights.

Prints ONE JSON line (rank 0): value = device-resident throughput (inputs already in HBM), e2e = the same metric with
the step's inputs copied from pinned host memory and the losses read back every step, roofline for the implicit-GEMM
convolution kernels (tensor bound), cpu_baseline = the reference algorithm (oracle port, fp32 PyTorch) on the host
cores. `--impl reference` times that CPU implementation alone (the reference has no GPU kernels of its own).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "train_images_per_sec"
UNIT = "images/s"
GF_PER_IMAGE_NECESSARY = 134.7   # conv+linear GFLOP per image of the necessary-work step (BASELINE.md section 3)



def workload_name(branches, batch):
    """The same string on both arms (the driver compares their `config`)."""
    return (f"birds_3stages.yml {branches}-stage 256x256 train step (G + D64/D128/D256 fwd+bwd, Adam, EMA), "
            f"batch {batch}/GPU")

def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps (with --sustain: at least this many)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"],
                    help="reference: the train step on the host CPU, the unmodified reference when a checkout of it is "
                         "given with $SG2_REF or placed at baseline/_ref (kind 'reference'), else the oracle port "
                         "(kind 'port'); its steps take seconds each, so raise SG2_BENCH_WATCHDOG for long runs")
    ap.add_argument("--batch", type=int, default=24, help="per-GPU batch (birds_3stages.yml: 24)")
    ap.add_argument("--branches", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--mode", default="train", choices=["train", "synth"],
                    help="train: the 3-stage train step (configs[1] / [2] / [4]); synth: generator-only eval-mode synthesis "
                         "from speech embeddings (configs[3], eval_birds.yml; use --batch 256)")
    ap.add_argument("--sustain", type=float, default=0.0,
                    help="keep replaying the step for at least this many seconds before / as the timed region (clocks and "
                         "power settle to the sustained state MEASURED_PEAKS.json's sustained figures refer to)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"], help="fp32: the fp32-accurate mode")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (rank 0; "
                         "train: losses and the updated weights, EMA weights and BatchNorm buffers; synth: the images), "
                         "each array larger than 2^20 elements as a fixed, seeded sample of 2^20 of its elements; "
                         "not with --sustain, whose step count depends on a measured step time")
    args = ap.parse_args()
    if args.dump_outputs and args.sustain > 0:
        ap.error("--dump-outputs needs a fixed number of steps: leave out --sustain")
    return args


def load_peaks(sustained):
    """-> (tensor peak TF/s, HBM GB/s, source). The conv replay of the roofline runs for tens of milliseconds at boost
    clocks: the BURST bf16 figure is its denominator; a --sustain run (seconds to minutes, ~1 kW) uses the sustained one."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        if sustained:
            return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json, sustained)"
        return d.get("bf16_tflops", 1650.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json, burst)"
    return (1400.0 if sustained else 1650.0), 6650.0, "fallback (B200_PROFILING.md)"


def dram_traffic_record():
    """ncu `dram__bytes_read.sum + dram__bytes_write.sum` of the dominant conv kernel family, per launch, from the committed
    capture (profiles/r02_conv_dram_traffic.json, written by tools/ncu_traffic.py); None when no capture is committed."""
    p = os.path.join(ROOT, "profiles", "r02_conv_dram_traffic.json")
    if not os.path.exists(p):
        return None
    try:
        return json.load(open(p))
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, pw = [], None, set(), []
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
                if len(f) > 6:
                    pw.append(float(f[6]))
            except ValueError:
                continue
            for name, val in zip(self.NAMES, f[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_median": statistics.median(pw) if pw else None}


# ------------------------------------------------------------------------------------------------ reference arm
def cpu_step_times(batch, branches, steps, warmup, threads):
    """The reference's CPU implementation of the train step on the host cores, fp32 PyTorch/oneDNN: the UNMODIFIED
    reference (condGANTrainer.train_Dnet / train_Gnet on its own G_NET / D_NET*) when a reference tree is available
    ($SG2_REF or baseline/_ref: oracle/ref_loader.py), else the oracle port of the same algorithm.
    -> (per-step seconds, kind)"""
    from oracle import ref_loader
    from oracle.stackgan_oracle import Cfg, OracleTrainer, synthetic_batch
    torch.set_num_threads(threads)
    cfg = Cfg(BRANCH_NUM=branches)
    torch.manual_seed(0)
    if ref_loader.reference_available():
        stepper, kind = ref_loader.ReferenceStepper(cfg, batch), "reference"
    else:
        stepper, kind = OracleTrainer(cfg), "port"
    times = []
    for s in range(warmup + steps):
        b = synthetic_batch(cfg, batch, seed=1234 + s)
        t0 = time.perf_counter()
        stepper.step(b)
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
    return times, kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.mode != "train":
        print(json.dumps({"impl": "reference", "unavailable": "the reference arm times the train step (configs[1]); "
                          "synthesis has no CPU reference leg"}))
        return
    cores = os.cpu_count() or 1
    steps, warmup = args.steps, args.warmup
    times, kind = cpu_step_times(args.batch, args.branches, steps, warmup, cores)
    ms = 1000.0 * sum(times) / len(times)
    value = args.batch / (ms / 1000.0)
    what = ("the unmodified reference (StackGAN_v2/model.py + trainer.py train_Dnet / train_Gnet)" if kind == "reference"
            else "oracle port of the reference (no reference checkout: set SG2_REF)")
    sample = (f"{steps} steps (+{warmup} warm-up) of the {args.branches}-stage train step at batch {args.batch}, {what}, "
              f"fp32 PyTorch CPU, {cores} threads")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.branches, args.batch), "global_batch": args.gpus * args.batch,
                   "parallelism": f"dp{args.gpus}"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------ our arm
DUMP_CAP = 1 << 20        # elements per dumped array: at most 10 arrays x 4 MB


def dump_outputs(out_dir, arrays):
    """Write each tensor, flattened, as out_dir/<name>.npy (float32; float64 stays float64). A tensor of more than DUMP_CAP
    elements is replaced by DUMP_CAP of its elements at positions fixed by its size (the same on every run and build)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().reshape(-1)
        if t.numel() > DUMP_CAP:
            idx = np.sort(np.random.default_rng([1234, t.numel()]).choice(t.numel(), DUMP_CAP, replace=False))
            t = t[torch.from_numpy(idx).to(t.device)]
        t = t.double() if t.dtype == torch.float64 else t.float()
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def step_outputs(tr, netG, netsD):
    """What one train step hands back to its caller: the loss vector [errD_0.., errG_total, kl, cal] and the networks it
    updated (parameters in the reference's order and OIHW shapes, the EMA copy of G's, floating-point buffers)."""
    flat = lambda ts: torch.cat([t.detach().reshape(-1).float() for t in ts])
    out = {"losses": tr.losses, "G_params": flat(netG.parameters()), "G_ema_params": flat(tr.bG.ema_params()),
           "G_buffers": flat(b for b in netG.buffers() if b.is_floating_point())}
    for i, d in enumerate(netsD):
        out[f"D{i}_params"] = flat(d.parameters())
        out[f"D{i}_buffers"] = flat(b for b in d.buffers() if b.is_floating_point())
    return out


def _shutdown(world, sdist):
    """Leave cleanly. destroy_process_group() used to block forever while CUDA graphs holding captured NCCL collectives
    were alive: the graphs are released first (callers delete them), the group is destroyed on a watchdog, and only if
    that still does not return within 20 s the process hard-exits (stdout already flushed)."""
    import torch.distributed as dist
    sys.stdout.flush()
    sys.stderr.flush()
    if world <= 1 or not dist.is_initialized():
        return
    done = threading.Event()

    def watchdog():
        if not done.wait(20.0):
            os._exit(0)

    threading.Thread(target=watchdog, daemon=True).start()
    try:
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
    finally:
        done.set()


def run_ours(args):
    import gc
    import torch.distributed as dist
    from sg2b200 import config, dist as sdist, ops, trainer, utils
    rank, local, world = sdist.init_from_env()
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("for --gpus N > 1 launch with: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    config.set_precision(args.precision)
    cfg = config.cfg
    cfg.TREE.BRANCH_NUM = args.branches
    B = args.batch
    torch.manual_seed(1234)
    netG, netsD = utils.build_networks(cfg, dev)
    sdist.broadcast_state([netG] + netsD)
    synth = args.mode == "synth"
    n_host = 3
    host = [utils.synthetic_batch(cfg, B, seed=1234 + 97 * rank + i, device="cpu", pin=True) for i in range(n_host)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    if synth:
        # ---- configs[3]: eval-mode generator-only synthesis from speech embeddings (trainer.py:681-803 evaluate())
        netG.eval()
        eng = netG.engine()
        eng.set_auto_refresh(False)          # weights are fixed: pack once, not on every no_grad forward
        for op in eng.conv_ops():
            op.packs()
        zs = torch.zeros(B, cfg.GAN.Z_DIM, device=dev)
        embs = torch.zeros(B, cfg.TEXT.DIMENSION, device=dev)
        epss = torch.zeros(B, cfg.GAN.EMBEDDING_DIM, device=dev)
        devb = [{k: hb[k].to(dev) for k in ("z", "emb")} for hb in host]

        def fwd():
            epss.normal_()                                   # model.py:190-193
            imgs, _, _, _ = eng.forward(zs, embs, epss, False)
            return imgs

        for _ in range(2):
            fwd()
        torch.cuda.synchronize()
        graph, n0 = None, ops.launches()
        if not args.no_graph:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out_imgs = fwd()
        else:
            out_imgs = fwd()
        per_step_launches = ops.launches() - n0

        def step_resident(i):
            nonlocal out_imgs
            b = devb[i % n_host]
            zs.copy_(b["z"], non_blocking=True)
            embs.copy_(b["emb"], non_blocking=True)
            if graph is not None:
                graph.replay()
            else:
                out_imgs = fwd()

        img_host = torch.empty(out_imgs[-1].shape, dtype=torch.float32).pin_memory()

        def step_e2e(i):
            hb = host[i % n_host]
            zs.copy_(hb["z"], non_blocking=True)             # pinned host -> device
            embs.copy_(hb["emb"], non_blocking=True)
            if graph is not None:
                graph.replay()
            else:
                fwd()
            img_host.copy_(out_imgs[-1], non_blocking=True)  # the product of synthesis: the 256 x 256 images, to the host

        h2d_bytes = sum(host[0][k].numel() * 4 for k in ("z", "emb"))
        d2h_bytes = img_host.numel() * 4
        step_eager, cap, tr = (lambda i: fwd()), None, None
        gf_per_image = 15.8186
    else:
        # one NCCL communicator per network (3 discriminators + G): their reductions are independent branches of the step
        reducer = sdist.GradAllReducer(channels=int(os.environ.get("SG2_COMMS", "4"))) if world > 1 else None
        tr = trainer.FusedTrainer(netG, netsD, cfg, all_reduce=reducer)
        devb = [{k: ([t.to(dev) for t in v] if isinstance(v, list) else v.to(dev)) for k, v in hb.items()} for hb in host]
        h2d_bytes = sum(t.numel() * t.element_size() for k, v in host[0].items() if k != "z"
                        for t in (v if isinstance(v, list) else [v]))
        d2h_bytes = tr.losses.numel() * 4
        noise = torch.empty(B, cfg.GAN.Z_DIM, device=dev)
        cap = None
        if not args.no_graph:
            cap = trainer.CapturedStep(tr, B)
            cap.load(devb[0]["emb"], devb[0]["real"], devb[0]["wrong"], devb[0]["labels"])
            cap.capture()
        per_step_launches = cap.launches_per_step if cap is not None else None

        def step_eager(i):
            b = devb[i % n_host]
            noise.normal_(0, 1)                                       # trainer.py:542
            return tr.step(noise, b["emb"], b["real"], b["wrong"], b["labels"])

        def step_resident(i):
            if cap is None:
                return step_eager(i)
            b = devb[i % n_host]
            cap.load(b["emb"], b["real"], b["wrong"], b["labels"])    # device -> static buffers (on-device copy)
            return cap.replay()

        # e2e: pinned host -> device copies of every step's inputs (copy stream, double buffered) + loss readback
        copy_stream = torch.cuda.Stream(device=dev)
        slots = [{k: ([torch.empty_like(t, device=dev) for t in v] if isinstance(v, list) else torch.empty_like(v, device=dev))
                  for k, v in host[0].items() if k != "z"} for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        loss_host = [torch.empty(tr.losses.numel(), dtype=torch.float32).pin_memory() for _ in range(2)]
        loss_ev = [torch.cuda.Event() for _ in range(2)]

        def prefetch(i):
            s_, hb = i % 2, host[i % n_host]
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[s_])
                for k, v in slots[s_].items():
                    if isinstance(v, list):
                        for d, h in zip(v, hb[k]):
                            d.copy_(h, non_blocking=True)
                    else:
                        v.copy_(hb[k], non_blocking=True)
                ready[s_].record(copy_stream)

        def step_e2e(i):
            if i == 0:
                prefetch(0)
            prefetch(i + 1)
            s_ = i % 2
            cur = torch.cuda.current_stream()
            cur.wait_event(ready[s_])
            b = slots[s_]
            if cap is None:
                noise.normal_(0, 1)
                losses = tr.step(noise, b["emb"], b["real"], b["wrong"], b["labels"])
            else:
                cap.load(b["emb"], b["real"], b["wrong"], b["labels"])
                losses = cap.replay()
            consumed[s_].record(cur)
            loss_host[s_].copy_(losses, non_blocking=True)
            loss_ev[s_].record(cur)
            if i > 0:
                loss_ev[1 - s_].synchronize()                         # the previous step's losses are on the host now
                _ = float(loss_host[1 - s_][0])

        for ev in consumed:
            ev.record(torch.cuda.current_stream())
        gf_per_image = GF_PER_IMAGE_NECESSARY

    for i in range(max(3, args.warmup)):
        step_resident(i)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    steps = args.steps
    if args.sustain > 0:
        # settle: replay for `sustain` seconds, then time the same number of seconds' worth of steps
        t_probe = timed(step_resident, 10) / 10.0
        steps = max(args.steps, int(1000.0 * args.sustain / t_probe))
        timed(step_resident, steps)
    l0 = ops.launches()
    ms_total = timed(step_resident, steps)
    launches = (ops.launches() - l0) if per_step_launches is None or args.no_graph else per_step_launches * steps
    clocks = sampler.stop() if rank == 0 else None
    ms_step = ms_total / steps
    value = world * B / (ms_step / 1000.0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {f"images{i}": im for i, im in enumerate(out_imgs)} if synth
                     else step_outputs(tr, netG, netsD))

    step_e2e(0)
    torch.cuda.synchronize()
    e2e_steps = min(steps, 200)
    ms_e2e = timed(step_e2e, e2e_steps) / e2e_steps
    e2e_value = world * B / (ms_e2e / 1000.0)

    # ---- roofline of the dominant kernel family (tcgen05 implicit-GEMM convolutions: fprop + dgrad + wgrad).
    # One eager step is run with call recording on; exactly those conv launches (same operands, same order) are then
    # replayed back to back inside one CUDA graph and timed with CUDA events: kernel time without host launch gaps and
    # without the elementwise kernels in between. achieved = executed MMA FLOPs of those launches / that time.
    peak_tf, peak_gbs, peak_src = load_peaks(sustained=False)
    roofline = None
    if not args.no_roofline:
        torch.cuda.synchronize()
        ops.profile_begin()
        step_eager(0)
        torch.cuda.synchronize()
        calls, keep = ops.profile_end()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for name, cargs, _ in calls:
                ops.replay_call(name, cargs)
        g.replay()
        torch.cuda.synchronize()
        reps = 5
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        conv_ms = e0.elapsed_time(e1) / reps
        flops = sum(c[2] for c in calls)
        del keep, g
        fam = {}
        for name, _, fl in calls:
            k = name.replace("sg2_conv_", "")
            fam[k] = fam.get(k, 0) + 1
        ach = flops / (conv_ms / 1000.0) / 1e12
        # The timed step overlaps its branches on several streams, so conv time / step time is not a share. For a
        # number comparable with the (serialised) ncu launch list, the same step is captured once more with every
        # kernel on ONE stream and timed: share_of_step = conv kernel time / serial kernel time of the step.
        serial_ms = None
        if world == 1 and cap is not None:
            was_concurrent = tr.concurrent
            try:
                tr.concurrent = False
                cap_s = trainer.CapturedStep(tr, B, warmup=1)
                cap_s.load(devb[0]["emb"], devb[0]["real"], devb[0]["wrong"], devb[0]["labels"])
                cap_s.capture()
                for _ in range(2):
                    cap_s.replay()
                torch.cuda.synchronize()
                e0.record()
                for _ in range(reps):
                    cap_s.replay()
                e1.record()
                torch.cuda.synchronize()
                serial_ms = e0.elapsed_time(e1) / reps
                del cap_s
            finally:
                tr.concurrent = was_concurrent
        elif synth:
            serial_ms = ms_step          # the synthesis forward is one stream
        traffic = dram_traffic_record()
        roofline = {"bound": "tensor",
                    "kernel": "tile_conv_kernel / tile_wgrad_kernel / igemm_fprop_kernel / igemm_wgrad_kernel "
                              "(every conv fprop + dgrad + wgrad launch of one step)",
                    "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                    "traffic": (traffic or {}).get("dram_bytes_per_launch"),
                    "traffic_detail": traffic,
                    "peak_source": peak_src + "; the conv replay is a ~30 ms burst at boost clocks",
                    "launches_per_step": len(calls), "launches_by_kind": fam,
                    "avg_launch_us": 1000.0 * conv_ms / max(1, len(calls)), "conv_ms_per_step": conv_ms,
                    "share_of_step": (conv_ms / serial_ms) if serial_ms else None,
                    "serial_step_ms": serial_ms, "conv_ms_over_overlapped_step_ms": conv_ms / ms_step,
                    "timing": "CUDA-graph replay of the recorded conv launches of one step, CUDA events, 5 replays; "
                              "share_of_step = that time / the same step captured on a single stream (no overlap)",
                    "flops_counting": "executed MMA FLOPs of each launch (fused-upsample convs run 4/9 of the reference's "
                                      "taps; padded channels of the 3-channel heads / stems are not counted)",
                    "step_tflops_reference_equivalent": gf_per_image * world * B / ms_step,
                    "step_frac_of_peak_reference_equivalent": gf_per_image * world * B / ms_step / (world * load_peaks(args.sustain > 0)[0])}

    # release every CUDA graph (they hold the captured NCCL collectives) before the process group goes away
    cap = None
    gc.collect()
    if rank != 0:
        _shutdown(world, sdist)
        return
    cpu = None
    if world == 1 and not args.no_cpu_baseline and not synth:
        cores = os.cpu_count() or 1
        t, kind = cpu_step_times(B, args.branches, 3, 1, cores)
        v = B / (sum(t) / len(t))
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": f"3 steps (+1 warm-up) of the {args.branches}-stage train step at batch {B} ("
                         + ("the unmodified reference" if kind == "reference" else "oracle port of the reference")
                         + ", fp32 PyTorch CPU)"}
    out = {
        "metric": METRIC if not synth else "synthesis_images_per_sec", "value": value, "unit": UNIT, "n_gpus": world,
        "steps": steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "f32 (3-way bf16 split on tcgen05, fp32 storage)",
        "data": "synthetic",
        "config": {"workload": workload_name(args.branches, B) if not synth else
                   f"eval_birds.yml generator-only {args.branches}-stage 256x256 synthesis from speech embeddings, batch {B}/GPU",
                   "global_batch": world * B, "parallelism": f"dp{world}"},
        "run": {"launch": "eager" if args.no_graph else "CUDA graph replay (whole step)",
                "l2": "inputs+activations per step (> 2 GB) exceed the 126 MB L2; no explicit flush",
                "sustain_s": args.sustain, "timed_seconds": ms_total / 1000.0, "precision": args.precision},
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": d2h_bytes},
        "gpu_launches": launches, "gpu_launches_per_step": launches / steps,
        "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
    }
    print(json.dumps(out))
    _shutdown(world, sdist)


def main():
    args = parse()
    # a run that stalls dumps every thread's Python stack and exits instead of hanging the caller (SG2_BENCH_WATCHDOG
    # seconds, default 600 + 4 x --sustain; the default run takes ~1 minute including the CPU baseline)
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("SG2_BENCH_WATCHDOG", str(int(600 + 4 * args.sustain)))), exit=True)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
