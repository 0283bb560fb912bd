"""Inception-v3 scorer measurements on one GPU (python tools/bench_inception.py [--out PATH]):

1. scorer forward, images/s at B = 48 (in-loop: 2 x 24) and B = 500 (snapshot batches): sg2b200.inception against
   torchvision's Inception3 in fp32 (TF32 off: the reference's arithmetic) and in bf16 autocast with channels_last. Arms
   alternate within the call; CUDA events after a warm-up; executed and useful MMA FLOP/s (torchvision: useful only).
2. the captured 3-stage train step at B = 24: ms/step without scoring, with scoring of fake and real, with scoring of
   the fake only; arms alternate, --replays per arm.

Prints the device name and power limit with the numbers and writes one JSON (default profiles/inception_bench.json).
Random weights: the timings do not depend on their values. A watchdog ends the process if the run hangs."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else None}


def time_arms(arms, rounds, iters):
    """arms: name -> callable. Alternating rounds of `iters` calls each; -> name -> median ms per call."""
    res = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                fn()
            b.record()
            b.synchronize()
            res[k].append(a.elapsed_time(b) / iters)
    return {k: sorted(v)[len(v) // 2] for k, v in res.items()}


def bench_forward(B, rounds, iters):
    import torchvision
    from sg2b200 import inception
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    ours = inception.INCEPTION_V3(random_init=True)
    tv = torchvision.models.inception_v3(weights=None, aux_logits=True, init_weights=False).cuda().eval()
    tv_cl = torchvision.models.inception_v3(weights=None, aux_logits=True, init_weights=False).cuda().eval()
    tv_cl = tv_cl.to(memory_format=torch.channels_last)
    img = torch.rand(B, 3, 256, 256, device="cuda") * 2 - 1

    def tv_in(x):
        x = x * 0.5 + 0.5
        m = torch.tensor([0.485, 0.456, 0.406], device="cuda").view(1, 3, 1, 1)
        s = torch.tensor([0.229, 0.224, 0.225], device="cuda").view(1, 3, 1, 1)
        return torch.nn.functional.interpolate((x - m) / s, size=(299, 299), mode="bilinear", align_corners=False)

    def f_tv():
        with torch.no_grad():
            return torch.softmax(tv(tv_in(img)), 1)

    def f_tv_bf16():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            return torch.softmax(tv_cl(tv_in(img).contiguous(memory_format=torch.channels_last)).float(), 1)

    arms = {"sg2b200": lambda: ours(img), "torchvision_fp32": f_tv, "torchvision_bf16_cl": f_tv_bf16}
    for fn in arms.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    ms = time_arms(arms, rounds, iters)
    rep = inception.utilisation_report(B)
    useful = 2.0 * B * sum(r["macs"] for r in rep)
    executed = 2.0 * sum(r["issued_rows"] * r["issued_cols"] * r["cin"] * r["kh"] * r["kw"] for r in rep)
    out = {}
    for k, t in ms.items():
        out[k] = {"ms": t, "images_per_s": B / t * 1e3, "useful_tflops": useful / t / 1e9,
                  "executed_tflops": executed / t / 1e9 if k == "sg2b200" else None}
    return out


def bench_step(replays, rounds):
    from oracle.stackgan_oracle import Cfg  # noqa: F401  (the parity helpers build the trainer from its config)
    from tests.parity_util import build_trainer_and_oracles, train_batch
    from sg2b200 import inception, trainer
    B = 24
    cfg, _, _, _, tr, _ = build_trainer_and_oracles(3, seed=0, n_oracles=0)
    b = train_batch(cfg, B, 1)
    scorer = inception.INCEPTION_V3(random_init=True)
    caps = {}
    for name, sc, real in (("no_scoring", None, True), ("score_fake_real", scorer, True), ("score_fake", scorer, False)):
        cap = trainer.CapturedStep(tr, B, warmup=2, scorer=sc, score_real=real)
        cap.load(b["emb"], b["real"], b["wrong"], b["labels"])
        caps[name] = cap.capture()
    for cap in caps.values():
        for _ in range(5):
            cap.replay()
    torch.cuda.synchronize()
    ms = time_arms({k: c.replay for k, c in caps.items()}, rounds, replays // rounds)
    return {k: {"ms_per_step": v, "replays": replays} for k, v in ms.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "inception_bench.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--replays", type=int, default=250, help="timed replays per captured-step arm")
    ap.add_argument("--watchdog", type=float, default=900.0, help="seconds before the process is ended")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_inception: no CUDA device")
    timer = threading.Timer(a.watchdog, lambda: (print("bench_inception: watchdog expired", flush=True), os._exit(3)))
    timer.daemon = True
    timer.start()
    import __graft_entry__
    __graft_entry__.build()
    t0 = time.time()
    res = {**device_info()}
    res["forward"] = {f"B{B}": bench_forward(B, a.rounds, it) for B, it in ((48, 10), (500, 2))}
    res["captured_step_B24_3stages"] = bench_step(a.replays, a.rounds)
    res["wall_s"] = time.time() - t0
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)
    print(json.dumps(res, indent=1))
    timer.cancel()


if __name__ == "__main__":
    main()
