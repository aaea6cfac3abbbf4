#!/usr/bin/env python
"""bench.py -- DSMIL aggregator forward throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

metric  : patches/sec of the DSMIL forward (MILNet.forward, dsmil.py:70-74) at N=10 000, D=512, C=2.
step    : one pass over a stream of `--bags` synthetic bags (default 16 x 10 000 x 512 fp32 = 328 MB,
          larger than the 126 MB L2, so every bag is read from HBM: "inputs larger than L2").
N GPUs  : weak scaling -- every bag is a giant bag of 10 000*N rows row-sharded over the N ranks
          (each rank keeps 10 000 rows per bag); two NCCL all-gathers per step carry the per-class
          critical-instance candidates and the softmax/partial-sum records (SURVEY §8e).
value   : whole-job patches/sec, inputs resident in HBM, CUDA-event timed, max over ranks.
e2e     : same metric through the public host-buffer API (dsmil_wsi_b200.pipeline.HostBagPipeline):
          pinned host bags -> H2D -> forward -> D2H of (classes, prediction_bag, A, B), per step.
roofline: frac = algorithmic bytes of the WHOLE forward step / CUDA-event step time / measured HBM peak
          (MEASURED_PEAKS.json); `dominant_kernel_frac` is the same bytes over the dominant kernel alone;
          `tensor_fraction` = bf16 tensor FLOPs issued (3xBF16: 3 products per GEMM) / step time / measured peak.
cpu_baseline: the reference's own MILNet (oracle/_ref/dsmil.py, staged unmodified by build(); kind
          "reference") or, when not staged, the oracle's torch-CPU port (kind "port") on a bounded sample.
extras  : torch_eager_gpu (the unmodified reference module through PyTorch eager on the same GPU = the kernel
          to beat), single-call milnet(x) latency, N=8 192 forward, N=15 000 C=1 forward+backward+Adam
          (train_tcga.py:67-73), and the N=100 000 giant-bag STRONG-scaling workload (BASELINE configs 1,2,4).
`--impl reference` times the reference's CPU implementation alone.
"""
import argparse
import contextlib
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

D, C, NBAG = 512, 2, 10000
METRIC = "patches/sec DSMIL fwd at N=10k D=512"


def algorithmic_bytes_fwd(N, D_, C_):
    """SURVEY §8(d): one read of X, write classes + A, weights once, B and pred."""
    W = 4 * (C_ * D_ + C_ + 128 * D_ + 128 + 128 * 128 + 128 + C_ * C_ * D_ + C_)
    return N * (4 * D_ + 8 * C_) + W + 4 * C_ * D_ + 4 * C_


def tensor_flops_fwd(N, D_, issued=True):
    """bf16 tensor-core FLOPs of the Q-MLP for N rows: 2*N*(D*128 + 128*128), x3 for the three split products
    the kernel issues (hi*Whi + lo*Whi + hi*Wlo)."""
    return (3 if issued else 1) * 2.0 * N * (D_ * 128 + 128 * 128)


def load_reference_module():
    """The UNMODIFIED reference dsmil.py staged in oracle/_ref (bench baseline legs only)."""
    try:
        from oracle import stage_ref
        return stage_ref.load_reference_dsmil()
    except Exception:
        return None


def make_reference_net(refmod, p, device, D_=None, C_=None):
    """Reference MILNet(FCLayer, BClassifier) holding the benchmark weights (or random init for other shapes)."""
    D_, C_ = D_ or D, C_ or C
    net = refmod.MILNet(refmod.FCLayer(D_, C_), refmod.BClassifier(D_, C_))
    if p is not None:
        t = lambda a: torch.from_numpy(np.array(a, dtype=np.float32))
        net.load_state_dict({"i_classifier.fc.0.weight": t(p.Wi), "i_classifier.fc.0.bias": t(p.bi),
                             "b_classifier.q.0.weight": t(p.W1), "b_classifier.q.0.bias": t(p.b1),
                             "b_classifier.q.2.weight": t(p.W2), "b_classifier.q.2.bias": t(p.b2),
                             "b_classifier.fcc.weight": t(p.Wf), "b_classifier.fcc.bias": t(p.bf)})
    return net.to(device)


def cuda_time_ms(fn, reps, warm=3):
    """Mean CUDA-event time of fn() over `reps` calls on the current stream (after `warm` untimed calls)."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        pk = json.load(open(path))
        return float(pk["hbm_gbs"]), float(pk.get("bf16_tflops", 1590.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


def warmup_plan(world: int, warmup: int):
    """(fixed_steps, timed_seconds, extra_fixed_steps).  Under torchrun every step contains collectives, so the
    number of warm-up steps must be the same on all ranks: fixed counts only.  A single process may extend the
    warm-up by wall-clock time so that the clock sampler sees >= 0.6 s of load."""
    fixed = max(int(warmup), 3)
    return (fixed, 0.6, 0) if world == 1 else (fixed, 0.0, 512)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "window": "warm-up (0.6 s of identical steps at N=1, 512 steps under torchrun) + timed region, nvidia-smi -lms 100"}


class Weights:
    """Seeded nn.Linear-scale weights for the benchmark model (random init of the reference architecture)."""

    def __init__(self, seed=0, scale=2.0):
        rng = np.random.default_rng(seed)
        u = lambda shape, fan: (rng.uniform(-1, 1, size=shape) * scale / np.sqrt(fan)).astype(np.float32)
        self.Wi, self.bi = u((C, D), D), u((C,), D)
        self.W1, self.b1 = u((128, D), D), u((128,), D)
        self.W2, self.b2 = u((128, 128), 128), u((128,), 128)
        self.Wf, self.bf = u((C, C, D), C * D), u((C,), C * D)


def make_params(seed=0):
    return Weights(seed)


def oracle_params(w):
    """CPU-baseline legs only: hand the same weights to the oracle's torch-CPU port."""
    from oracle import dsmil_oracle as orc
    return orc.Params(w.Wi, w.bi, w.Wf, w.bf, w.W1, w.b1, w.W2, w.b2)


def make_net(p, device):
    import dsmil as mil
    net = mil.MILNet(mil.FCLayer(D, C), mil.BClassifier(D, C))
    t = lambda a: torch.from_numpy(np.array(a, dtype=np.float32))
    net.load_state_dict({"i_classifier.fc.0.weight": t(p.Wi), "i_classifier.fc.0.bias": t(p.bi),
                         "b_classifier.q.0.weight": t(p.W1), "b_classifier.q.0.bias": t(p.b1),
                         "b_classifier.q.2.weight": t(p.W2), "b_classifier.q.2.bias": t(p.b2),
                         "b_classifier.fcc.weight": t(p.Wf), "b_classifier.fcc.bias": t(p.bf)})
    return net.to(device).eval()


class CpuArm:
    """The reference's CPU implementation of the path: its own MILNet (oracle/_ref/dsmil.py, unmodified, eval +
    no_grad) when staged -- kind "reference" -- else the oracle's torch-CPU port -- kind "port"."""

    def __init__(self, p, threads):
        self.threads = threads
        torch.set_num_threads(threads)
        refmod = load_reference_module()
        if refmod is not None:
            self.kind = "reference"
            self.net = make_reference_net(refmod, p, "cpu").eval()
            self.what = "unmodified reference dsmil.MILNet (oracle/_ref/dsmil.py:64-74), torch-CPU fp32, eval + no_grad"
        else:
            from oracle import dsmil_oracle as orc
            self.kind = "port"
            self.port = orc.TorchPort(oracle_params(p), threads=threads)
            self.what = "torch-CPU fp32 port of dsmil.py:46-62 (oracle/dsmil_oracle.py TorchPort)"

    def forward(self, x):
        if self.kind == "reference":
            with torch.no_grad():
                return self.net(x)
        return self.port.forward(x)


def best_cpu_threads(p, bags, budget=0.6):
    """torch-CPU with one thread per core is NOT the fastest setting on a many-core host for ops this
    small; give the baseline the thread count it likes best (short calibration, reported as `cores`)."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu})
    best, best_rate = cands[0], 0.0
    for c in cands:
        arm = CpuArm(p, c)
        arm.forward(bags[0])
        t0 = time.perf_counter(); n = 0
        while time.perf_counter() - t0 < budget:
            arm.forward(bags[n % len(bags)]); n += 1
        rate = n / (time.perf_counter() - t0)
        if rate > best_rate:
            best, best_rate = c, rate
    return best


def cpu_port_rate(p, seconds, threads=None, nbags=16):
    """CPU arm on a bounded sample (distinct bags cycled, like the GPU arm's step): returns patches/s."""
    g = torch.Generator().manual_seed(1)
    bags = [torch.rand(NBAG, D, generator=g) for _ in range(nbags)]
    threads = threads or best_cpu_threads(p, bags[:4])
    arm = CpuArm(p, threads)
    for b in bags[:2]:
        arm.forward(b)
    t0 = time.perf_counter()
    n = 0
    while time.perf_counter() - t0 < seconds:
        arm.forward(bags[n % nbags])
        n += 1
    dt = time.perf_counter() - t0
    return n * NBAG / dt, arm, n


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores -- the unmodified
    reference module staged in oracle/_ref when present (kind "reference"), else the oracle port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    g = torch.Generator().manual_seed(1)
    nb = args.ref_bags
    bags = [torch.rand(NBAG, D, generator=g) for _ in range(nb)]
    arm = CpuArm(make_params(), best_cpu_threads(make_params(), bags[:4]))
    for _ in range(max(args.warmup, 1)):
        for b in bags:
            arm.forward(b)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for b in bags:
            arm.forward(b)
    dt = time.perf_counter() - t0
    val = args.steps * nb * NBAG / dt
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "patches/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"stream of {nb} synthetic bags, each N={NBAG} x D={D}, C={C}, DSMIL forward "
                                  "(bounded sample of the GPU arm's 16-bag step)", "bags_per_step": nb},
           "cpu_baseline": {"value": val, "unit": "patches/s", "cores": arm.threads, "kind": arm.kind,
                            "sample": f"{args.steps} steps x {nb} bags x {NBAG} patches; {arm.what}; all host threads "
                                      f"it scales to ({arm.threads})"},
           "e2e": {"value": val, "unit": "patches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def run_extras(args, p, net, bags, dev, ms_per_step):
    """Rank 0, one GPU: the other BASELINE configs and the 'kernel to beat' (same box, same run)."""
    import dsmil as mil
    ex = {}
    refmod = load_reference_module()
    nb = len(bags)
    # (1) the unmodified reference module through PyTorch eager on this GPU, same bags, same weights
    if refmod is not None:
        rnet = make_reference_net(refmod, p, dev).eval()

        def eager_step():
            with torch.no_grad():
                for b in bags:
                    rnet(b)
        ms = cuda_time_ms(eager_step, 5, warm=2)
        ex["torch_eager_gpu"] = {"value": nb * NBAG / (ms / 1e3), "unit": "patches/s", "ms_per_step": ms,
                                 "what": "oracle/_ref/dsmil.py MILNet (unmodified reference), eval + no_grad, PyTorch eager "
                                         "on cuda:0, same 16 bags and weights", "speedup_device_timed": ms / ms_per_step}
    else:
        rnet = None
        ex["torch_eager_gpu"] = {"unavailable": "reference sources not staged in oracle/_ref"}
    # (2) the call the reference's drivers make: ONE bag through milnet(x)  (train_tcga.py:98)
    with torch.no_grad():
        one = cuda_time_ms(lambda: net(bags[0]), 50, warm=5)
        ex["single_call_n10000"] = {"ms": one, "patches_per_s": NBAG / (one / 1e3), "api": "milnet(x), eval, no_grad"}
        if rnet is not None:
            r1 = cuda_time_ms(lambda: rnet(bags[0]), 20, warm=3)
            ex["single_call_n10000"].update({"torch_eager_gpu_ms": r1, "speedup": r1 / one})
    # (3) BASELINE configs[1]: N=8 192 forward
    g = torch.Generator(device=dev).manual_seed(7)
    b8 = [torch.rand(8192, D, generator=g, device=dev) for _ in range(nb)]
    with torch.no_grad():
        ms8 = cuda_time_ms(lambda: net.forward_bags(b8), 20, warm=3)
    ex["fwd_n8192"] = {"value": nb * 8192 / (ms8 / 1e3), "unit": "patches/s", "ms_per_step": ms8, "bags_per_step": nb,
                       "hbm_frac": algorithmic_bytes_fwd(8192, D, C) * nb / (ms8 / 1e3) / 1e9 / load_peaks()[0]}
    del b8
    # (4) BASELINE configs[2]: Camelyon16 shape, N=15 000, C=1, forward + backward + Adam (train_tcga.py:67-73,232)
    NT, CT_ = 15000, 1
    tb = [torch.rand(NT, D, generator=g, device=dev) for _ in range(4)]
    lab = torch.ones(1, CT_, device=dev)

    def make_train(modlib):
        torch.manual_seed(0)
        m = modlib.MILNet(modlib.FCLayer(D, CT_), modlib.BClassifier(D, CT_)).to(dev).train()
        opt = torch.optim.Adam(m.parameters(), lr=1e-4, betas=(0.5, 0.9), weight_decay=1e-3)
        crit = torch.nn.BCEWithLogitsLoss()
        k = [0]

        def tstep():
            opt.zero_grad()
            ins, bagp, _, _ = m(tb[k[0] % 4]); k[0] += 1
            mx, _ = torch.max(ins, 0)
            loss = 0.5 * crit(bagp.view(1, -1), lab) + 0.5 * crit(mx.view(1, -1), lab)
            loss.backward()
            opt.step()
        return tstep
    mst = cuda_time_ms(make_train(mil), 20, warm=3)
    ex["train_n15000_c1"] = {"ms_per_step": mst, "patches_per_s": NT / (mst / 1e3), "slides_per_s": 1e3 / mst,
                             "what": "milnet(x) -> 0.5*BCE(bag)+0.5*BCE(max) -> backward -> Adam, one bag per step"}
    if refmod is not None:
        msr = cuda_time_ms(make_train(refmod), 10, warm=3)
        ex["train_n15000_c1"].update({"torch_eager_gpu_ms": msr, "speedup": msr / mst})
    # (5) the embedder of compute_feats.py:146-174: torchvision ResNet-18 with InstanceNorm2d + fc, batch 128 x 3 x 224 x 224
    try:
        ex["embed_resnet18_in"] = embed_leg(dev, refmod)
    except Exception as e:                                    # torchvision missing etc.: report, do not fail the bench
        ex["embed_resnet18_in"] = {"unavailable": f"{type(e).__name__}: {str(e)[:160]}"}
    # (6) the patch loader + the whole compute_feats loop from JPEG FILES on disk (compute_feats.py:19-82)
    try:
        ex["embed_from_files"] = files_leg(dev, refmod)
    except Exception as e:
        ex["embed_from_files"] = {"unavailable": f"{type(e).__name__}: {str(e)[:160]}"}
    return ex


def synth_patch_files(n, seed=0, hw=224, quality=70):
    """n JPEG files shaped like the reference's patches (deepzoom_tiler.py saves 224 x 224 tiles with PIL, quality 70,
    PIL defaults = 4:2:0, standard Huffman tables): smooth stained-tissue-like blobs + noise, not white noise."""
    import io
    from PIL import Image
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:hw, 0:hw].astype(np.float32)
    out = []
    for _ in range(n):
        img = np.zeros((hw, hw, 3), np.float32) + np.array([225.0, 190.0, 215.0], np.float32)
        for _ in range(12):
            cy, cx, r = rng.uniform(0, hw), rng.uniform(0, hw), rng.uniform(3, hw / 4)
            img -= np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2 * r * r))[..., None] * rng.uniform(30, 140, 3).astype(np.float32)
        img += rng.normal(0, 6, img.shape).astype(np.float32)
        b = io.BytesIO()
        Image.fromarray(np.clip(img, 0, 255).astype(np.uint8)).save(b, format="JPEG", quality=quality)
        out.append(b.getvalue())
    return out


def files_leg(dev, refmod, n_files=4096, batch=128, workers=4, n_bags=2):
    """(a) the device JPEG loader alone on one 128-patch batch, against PIL on `workers` host threads (the reference's
    DataLoader(num_workers=4)); (b) compute_feats over a bag folder of n_files patches, wall clock, CSV written:
    this repo's loop (device decode / host decode) and the reference's own unmodified compute_feats.compute_feats."""
    import shutil
    import tempfile
    import types
    from concurrent.futures import ThreadPoolExecutor
    import dsmil as mil
    from dsmil_wsi_b200 import embed, jpeg
    from oracle import stage_ref
    distinct = synth_patch_files(batch, seed=5)
    out = {"what": f"{n_files} patch files in {n_bags} bag folders (224 x 224 JPEG, quality 70, PIL defaults; {batch} distinct images), batch {batch}, "
                   f"{workers} loader workers, ResNet-18-InstanceNorm embedder, '%.4f' CSV written",
           "bytes_per_file": int(np.mean([len(f) for f in distinct]))}
    # (a) loader alone
    pb = jpeg.parse_batch(distinct, pin=True)
    dec = jpeg.JpegBatchDecoder(dev)
    x = torch.empty(batch, 3, 224, 224, device=dev)
    ms = cuda_time_ms(lambda: dec.decode(pb, out_f32=x), 10, warm=2)
    st = dec.decode(pb, out_f32=x)
    torch.cuda.synchronize()
    if st.cpu().abs().sum().item() != 0:
        raise RuntimeError("device JPEG decode reported a failure")
    t0 = time.perf_counter()
    for _ in range(3):
        jpeg.parse_batch(distinct)
    parse_ms = (time.perf_counter() - t0) / 3 * 1e3
    with ThreadPoolExecutor(workers) as pool:
        list(pool.map(embed._decode_u8, distinct[:16]))
        t0 = time.perf_counter()
        ref_imgs = list(pool.map(embed._decode_u8, distinct))
        pil_ms = (time.perf_counter() - t0) * 1e3
    same = bool(np.array_equal((x[0].permute(1, 2, 0) * 255).round().byte().cpu().numpy(), ref_imgs[0]))
    out["loader_batch128"] = {"device_ms": ms, "device_patches_per_s": batch / (ms / 1e3), "host_parse_ms": parse_ms,
                              "pil_threads_ms": pil_ms, "pil_patches_per_s": batch / (pil_ms / 1e3), "threads": workers,
                              "speedup": pil_ms / ms, "first_patch_equals_pil": same,
                              "h2d_bytes_device_route": int(pb.blob_bytes + pb.n * jpeg.header_bytes()),
                              "h2d_bytes_reference": batch * 3 * 224 * 224 * 4,
                              "what": "H2D of the files + k_jpeg_entropy/idct/color (CUDA events) vs PIL decode on host threads"}
    # one launch over 8 batches: the entropy kernel is latency-bound per patch (one warp each), so its time does not grow
    pb8 = jpeg.parse_batch(distinct * 8, pin=True)
    x8 = torch.empty(8 * batch, 3, 224, 224, device=dev)
    ms8 = cuda_time_ms(lambda: dec.decode(pb8, out_f32=x8), 5, warm=2)
    out["loader_batch1024"] = {"device_ms": ms8, "device_patches_per_s": 8 * batch / (ms8 / 1e3)}
    del x8, pb8
    # (b) the loop from a folder
    root = tempfile.mkdtemp(prefix="dsmil_files_")
    try:
        bags = [os.path.join(root, "in", "class0", f"bag{b}") for b in range(n_bags)]
        for b, bag in enumerate(bags):
            os.makedirs(bag)
            for i in range(n_files // n_bags):
                with open(os.path.join(bag, f"{i // 32}_{i % 32}.jpeg"), "wb") as f:
                    f.write(distinct[(i + 7 * b) % batch])
        args = types.SimpleNamespace(batch_size=batch, num_workers=workers)
        ours = make_embedder(mil, dev, True)              # embed_bag switches it to channels-last itself

        def run(fn, route=None):
            if route is not None:
                os.environ["DSMIL_B200_JPEG"] = route
            best = None
            for rep in range(2):                         # first pass warms cuDNN / the page cache
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                with contextlib.redirect_stdout(sys.stderr):          # both loops print progress; stdout carries the JSON line
                    fn(os.path.join(root, f"out_{route}_{rep}"))
                torch.cuda.synchronize()
                best = time.perf_counter() - t0
            os.environ.pop("DSMIL_B200_JPEG", None)
            return best
        t_dev = run(lambda sp: embed.compute_feats(args, bags, ours, sp), "gpu")
        t_host = run(lambda sp: embed.compute_feats(args, bags, ours, sp), "host")
        out["compute_feats"] = {"value": n_files / t_dev, "unit": "patches/s", "seconds": t_dev,
                                "host_decode_route_patches_per_s": n_files / t_host, "host_decode_route_seconds": t_host}
        rcf = stage_ref.load_reference_compute_feats()
        if rcf is not None and refmod is not None:
            ref = make_embedder(refmod, dev, False)
            t_ref = run(lambda sp: rcf.compute_feats(args, bags, ref, sp, "single"))
            out["compute_feats"].update({"reference_patches_per_s": n_files / t_ref, "reference_seconds": t_ref,
                                         "speedup": t_ref / t_dev,
                                         "reference": "oracle/_ref/compute_feats.py compute_feats (unmodified): DataLoader workers + PIL "
                                                      "+ .float().cuda() + eager backbone + pandas CSV, same GPU"})
            a = open(os.path.join(root, "out_gpu_1", "class0", "bag0.csv")).read()
            b = open(os.path.join(root, "out_None_1", "class0", "bag0.csv")).read()
            fa = np.loadtxt(io_lines(a), delimiter=",", skiprows=1)
            fb = np.loadtxt(io_lines(b), delimiter=",", skiprows=1)
            out["compute_feats"]["max_abs_csv_diff_vs_reference"] = float(np.abs(fa - fb).max())
    finally:
        shutil.rmtree(root, ignore_errors=True)
    return out


def io_lines(text):
    import io
    return io.StringIO(text)


def make_embedder(modlib, dev, fuse, channels_last=False):
    import torchvision.models as models
    torch.manual_seed(0)
    resnet = models.resnet18(weights=None, norm_layer=torch.nn.InstanceNorm2d)    # compute_feats.py:154 (norm_layer='instance')
    for prm in resnet.parameters():
        prm.requires_grad = False
    resnet.fc = torch.nn.Identity()
    ic = modlib.IClassifier(resnet, 512, C).to(dev).eval()
    if fuse:
        from dsmil_wsi_b200.embedder import fuse_instance_norm
        fuse_instance_norm(ic.feature_extractor)
    if channels_last:                                     # what embed.embed_bag does to the backbone (DSMIL_B200_NHWC)
        ic.feature_extractor.to(memory_format=torch.channels_last)
    return ic


def embed_leg(dev, refmod, batch=128):
    import dsmil as mil
    g = torch.Generator(device=dev).manual_seed(3)
    x = torch.rand(batch, 3, 224, 224, generator=g, device=dev)
    out = {"batch": batch, "what": "IClassifier(ResNet-18 with nn.InstanceNorm2d, fc) on a 128 x 3 x 224 x 224 fp32 batch "
                                   "(compute_feats.py:70-76,146-174); convolutions = cuDNN in both arms (TF32 allowed, torch default)"}
    ours = make_embedder(mil, dev, True, channels_last=True)
    xcl = x.contiguous(memory_format=torch.channels_last)     # the layout the JPEG loader writes the batch in
    with torch.no_grad():
        ms = cuda_time_ms(lambda: ours(xcl), 5, warm=2)
        ours_nchw = make_embedder(mil, dev, True)
        ms_nchw = cuda_time_ms(lambda: ours_nchw(x), 5, warm=2)
        del ours_nchw
    out.update({"value": batch / (ms / 1e3), "unit": "patches/s", "ms_per_batch": ms, "ms_per_batch_nchw": ms_nchw,
                "ours": "channels-last: convs cuDNN NHWC; InstanceNorm + residual + ReLU fused (dsmil_instnorm_act_nhwc); fc "
                        "scores by libdsmil_b200.  ms_per_batch_nchw = the same with NCHW memory (dsmil_instnorm_act)"})
    if refmod is not None:
        ref = make_embedder(refmod, dev, False)
        with torch.no_grad():
            msr = cuda_time_ms(lambda: ref(x), 5, warm=2)
            fa, fb = ours(xcl)[0], ref(x)[0]
        out.update({"torch_eager_gpu_ms": msr, "torch_eager_gpu_patches_per_s": batch / (msr / 1e3), "speedup": msr / ms,
                    "max_abs_feature_diff": float((fa - fb).abs().max())})
    return out


def dump_outputs(out_dir, bag_outputs):
    """Writes what one forward_bags step hands its caller -- per bag (classes, prediction_bag, A, B) -- as float32
    arrays concatenated over the bags: classes.npy [sum N, C], prediction_bag.npy [bags, C], A.npy [sum N, C],
    B.npy [bags, C, D].  16 bags of N=10 000 come to 2.6 MB."""
    os.makedirs(out_dir, exist_ok=True)
    for i, name in enumerate(("classes", "prediction_bag", "A", "B")):
        t = torch.cat([o[i] for o in bag_outputs])
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def run_ours(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the DSMIL B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        # a collective that cannot complete (e.g. a rank died) aborts after 3 minutes instead of hanging the box
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    from dsmil_wsi_b200 import _lib
    from dsmil_wsi_b200.pipeline import HostBagPipeline
    from dsmil_wsi_b200.sharded import (CudaShardBagOps, CudaShardOps, ShardedBagsGraph, milnet_params,
                                        sharded_forward_bags, sharded_forward_bags_batched)
    lib = _lib.load()

    p = make_params()
    net = make_net(p, dev)
    nb = args.bags
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    bags = [torch.rand(NBAG, D, generator=g, device=dev) for _ in range(nb)]   # this rank's rows of each bag
    offsets = [rank * NBAG] * nb
    ops = bops = None
    if world > 1:
        if CudaShardBagOps.supported(milnet_params(net)):
            bops = CudaShardBagOps(milnet_params(net))
        else:
            ops = CudaShardOps(milnet_params(net))

    def sharded_step(xs):
        if bops is not None:
            return sharded_forward_bags_batched(bops, xs, offsets)
        return sharded_forward_bags(ops, xs, offsets)

    # the serving-loop form of the sharded step: one CUDA graph (3 library calls + 2 NCCL all-gathers) per step
    plan = None
    graph_note = "eager (host-launched)"
    if world > 1 and bops is not None and not args.no_graph:
        try:
            with torch.no_grad():
                plan = ShardedBagsGraph(bops, bags, offsets)
            graph_note = "CUDA graph replay (dsmil_wsi_b200.sharded.ShardedBagsGraph)"
        except Exception as e:                     # same code on every rank: the decision is collective
            plan = None
            graph_note = f"eager (graph capture failed: {type(e).__name__}: {str(e)[:120]})"

    def step():
        with torch.no_grad():
            if world == 1:
                return net.forward_bags(bags)
            if plan is not None:
                return plan.replay()
            return sharded_step(bags)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks / throttle reasons are sampled from the warm-up on (the timed region alone lasts a few ms, shorter
    # than nvidia-smi's fastest period).  The number of warm-up steps MUST be identical on every rank (each
    # step contains collectives), so it is a fixed count under torchrun and time-based only for a single process.
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    fixed_steps, timed_s, extra_steps = warmup_plan(world, args.warmup)
    for _ in range(fixed_steps):
        step()
    torch.cuda.synchronize()
    t_w = time.perf_counter()
    n_w = 0
    while time.perf_counter() - t_w < timed_s:        # single process only (timed_s == 0 under torchrun)
        step()
        n_w += 1
        if n_w % 8 == 0:
            torch.cuda.synchronize()
    for n_w in range(1, extra_steps + 1):              # same count on all ranks
        step()
        if n_w % 8 == 0:
            torch.cuda.synchronize()
    barrier()
    l0 = lib.dsmil_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        last = step()
    e1.record()
    barrier()
    launches = int(lib.dsmil_launch_count() - l0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
        del last
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = ms_total / args.steps
    patches_per_step = nb * NBAG * world
    value = patches_per_step / (ms_per_step / 1e3)

    # ---- roofline: whole forward step (headline) + the dominant kernel, timed live with CUDA events ----
    hbm_peak, tf_peak, peak_src = load_peaks()
    lib.dsmil_profile_enable(1)
    for _ in range(2):                             # host-launched here: graph replays carry no per-kernel event pairs
        with torch.no_grad():
            net.forward_bags(bags) if world == 1 else sharded_step(bags)
    torch.cuda.synchronize()
    ms_tag = (ctypes.c_double * 8)()
    n_tag = (ctypes.c_uint64 * 8)()
    lib.dsmil_profile_read(ms_tag, n_tag)
    lib.dsmil_profile_enable(0)
    tags = ["scores", "q_mlp", "attend", "finalize", "fused_sm100"]
    per = {t: (ms_tag[i] / n_tag[i] if n_tag[i] else None) for i, t in enumerate(tags)}
    dom = max((t for t in tags if per[t]), key=lambda t: per[t] * n_tag[tags.index(t)])
    launches_dom = int(n_tag[tags.index(dom)])
    bags_per_launch = 2.0 * nb / launches_dom          # 2 profiled steps of nb bags each
    alg_step = algorithmic_bytes_fwd(NBAG, D, C) * nb   # this rank's algorithmic bytes per step
    dom_ms = per[dom]
    achieved = alg_step / (ms_per_step / 1e3) / 1e9     # whole forward: every kernel and gap of the step is charged
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(tpath):     # dram__bytes_read+write of the step's kernels from the committed ncu --set full capture
        tj = json.load(open(tpath))
        traffic = tj.get("dram_bytes_per_step_16x10k")
        if traffic is not None and nb != 16:
            traffic = traffic * nb / 16.0
    tflops = tensor_flops_fwd(NBAG * nb, D) / (ms_per_step / 1e3) / 1e12
    roofline = {"bound": "hbm", "kernel": "whole forward step (all kernels of forward_bags)", "achieved": achieved,
                "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                "peak_source": peak_src, "algorithmic_bytes_per_step": alg_step,
                "dominant_kernel": dom, "dominant_kernel_ms": dom_ms,
                "dominant_kernel_frac": (algorithmic_bytes_fwd(NBAG, D, C) * bags_per_launch / (dom_ms / 1e3) / 1e9) / hbm_peak,
                "per_kernel_ms": {k: v for k, v in per.items() if v},
                "tensor_fraction": tflops / tf_peak, "tensor_tflops_issued": tflops, "tensor_peak_tflops": tf_peak,
                "tensor_fraction_algorithmic": tflops / 3.0 / tf_peak,
                "note": "frac = algorithmic bytes of the forward (SURVEY 8d: 2048+8C B/patch + weights, x bags per step) / "
                        "CUDA-event time of the whole step / measured HBM copy peak; dominant_kernel_frac charges only the "
                        "dominant kernel's duration; tensor_fraction = bf16 FLOPs issued (3 split products per GEMM) / step "
                        "time / measured bf16 peak (tensor_fraction_algorithmic counts each GEMM once)"}

    # ---- end to end through the public host-buffer API ------------------------------------------
    e2e = None
    if world == 1:
        host = [b.cpu().pin_memory() for b in bags]
        pipe = HostBagPipeline(net, NBAG, D, C)
        for _ in range(2):
            pipe.run(host)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps = max(2, min(args.steps, 10))
        for _ in range(reps):
            pipe.run(host)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / reps
        h2d, d2h = pipe.bytes_per_bag(NBAG)
        e2e = {"value": nb * NBAG / dt, "unit": "patches/s", "h2d_bytes_per_step": h2d * nb,
               "d2h_bytes_per_step": d2h * nb, "ms_per_step": dt * 1e3,
               "api": "dsmil_wsi_b200.pipeline.HostBagPipeline.run(pinned host bags)"}
    else:
        # multi-GPU e2e: every rank stages its shard from pinned host memory, then the sharded forward
        host = [b.cpu().pin_memory() for b in bags]
        slots = [torch.empty_like(b) for b in bags]
        outs_host = None

        def e2e_step():
            with torch.no_grad():
                for s, h in zip(slots, host):
                    s.copy_(h, non_blocking=True)
                outs = sharded_step(slots)
                return [tuple(t.cpu() for t in o[:4]) for o in outs]
        e2e_step(); barrier()
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            e2e_step()
        barrier()
        dt = torch.tensor([(time.perf_counter() - t0) / reps], device=dev)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dt = float(dt.item())
        e2e = {"value": patches_per_step / dt, "unit": "patches/s", "h2d_bytes_per_step": 4 * NBAG * D * nb * world,
               "d2h_bytes_per_step": 4 * (2 * NBAG * C + C + C * D) * nb * world, "ms_per_step": dt * 1e3,
               "api": "pinned host shards -> sharded_forward_bags -> host"}

    # ---- giant-bag STRONG scaling (BASELINE configs[4], north_star ">= 6x at 8 GPUs on N=100 000"): the SAME bags at
    # every world size, rows sharded over the ranks; value = total rows / max-over-ranks device time -------------
    strong = None
    if not args.no_extras:
        NG, nbg = 100000, args.giant_bags
        lo, hi = [(NG * r) // world for r in (rank, rank + 1)]
        gg = torch.Generator(device=dev).manual_seed(4242)
        giant = []
        for _ in range(nbg):        # every rank draws the full bag from the same seed and keeps its slice
            full = torch.rand(NG, D, generator=gg, device=dev)
            giant.append(full[lo:hi].clone())
            del full
        goff = [lo] * nbg

        gplan = None
        if plan is not None:                       # same decision on every rank
            try:
                with torch.no_grad():
                    gplan = ShardedBagsGraph(CudaShardBagOps(milnet_params(net)), giant, goff)
            except Exception:
                gplan = None

        def gstep():
            with torch.no_grad():
                if world == 1:
                    return net.forward_bags(giant)
                if gplan is not None:
                    return gplan.replay()
                if bops is not None:
                    return sharded_forward_bags_batched(bops, giant, goff)
                return sharded_forward_bags(ops, giant, goff)
        for _ in range(5):
            gstep()
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        greps = 20
        g0.record()
        for _ in range(greps):
            gstep()
        g1.record()
        barrier()
        gms = torch.tensor([g0.elapsed_time(g1) / greps], device=dev)
        if world > 1:
            dist.all_reduce(gms, op=dist.ReduceOp.MAX)
        gms = float(gms.item())
        galg = algorithmic_bytes_fwd(NG, D, C) * nbg
        strong = {"workload": f"{nbg} giant bags x N={NG} x D={D}, C={C}, rows sharded over {world} GPU(s) "
                              f"({hi - lo} rows/rank/bag); {nbg * NG * D * 4 / 1e6:.0f} MB of features in total (> L2)",
                  "scaling": "strong", "value": nbg * NG / (gms / 1e3), "unit": "patches/s", "ms_per_step": gms,
                  "n_gpus": world, "hbm_frac_per_gpu": galg / world / (gms / 1e3) / 1e9 / hbm_peak,
                  "step_launch": "CUDA graph replay" if gplan is not None else "eager"}
        del giant

    # ---- BASELINE configs[3]: ResNet-18 embedding of 224x224 patches + aggregator, patches sharded over the ranks ----
    embed_agg = None
    if not args.no_extras:
        try:
            import dsmil as mil
            from dsmil_wsi_b200.sharded import sharded_forward
            PB, NBATCH = 128, 4                       # 512 patches per rank per slide
            ic = make_embedder(mil, dev, True, channels_last=True)
            gen = torch.Generator(device=dev).manual_seed(50 + rank)
            px = [torch.rand(PB, 3, 224, 224, generator=gen, device=dev).contiguous(memory_format=torch.channels_last)
                  for _ in range(NBATCH)]
            sops = CudaShardOps(milnet_params(net)) if world > 1 else None

            def slide():
                with torch.no_grad():
                    feats = torch.cat([ic(b)[0] for b in px])             # [512, 512] on this rank
                    if world == 1:
                        return net(feats)
                    return sharded_forward(sops, feats, rank * PB * NBATCH)
            for _ in range(2):
                slide()
            barrier()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(3):
                slide()
            s1.record()
            barrier()
            tms = torch.tensor([s0.elapsed_time(s1) / 3], device=dev)
            if world > 1:
                dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            tms = float(tms.item())
            embed_agg = {"value": PB * NBATCH * world / (tms / 1e3), "unit": "patches/s", "ms_per_slide": tms,
                         "slides_per_s": 1e3 / tms, "patches_per_rank": PB * NBATCH, "n_gpus": world, "scaling": "weak",
                         "what": "per slide: each rank embeds its 512 patches (ResNet-18-InstanceNorm, channels-last, fused norm kernel) and the "
                                 "features go straight into the row-sharded DSMIL aggregator (NCCL: candidates + partial sums)"}
            del px, ic
        except Exception as e:
            embed_agg = {"unavailable": f"{type(e).__name__}: {str(e)[:160]}"}

    # ---- per-phase breakdown of one host-launched sharded step (CUDA events on the launch stream, max over ranks) -----
    breakdown = None
    if world > 1 and bops is not None and not args.no_extras:
        from dsmil_wsi_b200.sharded import _all_gather
        names = ["phase1 (scores+keys+Q-MLP+candidates)", "all_gather candidates", "phase2 (merge+attend+local record)",
                 "all_gather records", "phase3 (combine+normalise+bag logits)"]
        acc = [0.0] * 5
        reps_b = 10
        with torch.no_grad():
            for it_b in range(reps_b + 2):
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
                bops.begin(bags, offsets)
                ev[0].record(); cand = bops.phase1()
                ev[1].record(); cands_all, Gg = _all_gather(cand.view(-1), None)
                ev[2].record(); recs_l = bops.phase2(cands_all, Gg)
                ev[3].record(); recs_all, Gg = _all_gather(recs_l.view(-1), None)
                ev[4].record(); bops.phase3(recs_all, Gg)
                ev[5].record()
                torch.cuda.synchronize()
                if it_b >= 2:
                    for i in range(5):
                        acc[i] += ev[i].elapsed_time(ev[i + 1]) / reps_b
        tb = torch.tensor(acc, device=dev)
        dist.all_reduce(tb, op=dist.ReduceOp.MAX)
        breakdown = {"unit": "ms", "launch": "eager (host-launched), events between the five calls, max over ranks",
                     **{n: float(v) for n, v in zip(names, tb.tolist())}, "sum": float(tb.sum().item())}

    # ---- multi-rank parity check (outside every timed region): one sharded forward against the CPU oracle ------
    parity = None
    if world > 1 and not args.no_extras:
        from oracle import dsmil_oracle as orc
        Nc = 4096 * world + 37
        xc = orc.synthetic_bag(Nc, D, 9, "uniform")
        lo, hi = [(Nc * r) // world for r in (rank, rank + 1)]
        xl = torch.from_numpy(xc[lo:hi]).to(dev)
        with torch.no_grad():
            o = (sharded_forward_bags_batched(bops, [xl], [lo]) if bops is not None
                 else sharded_forward_bags(ops, [xl], [lo]))[0]
        t = orc.forward(xc, oracle_params(p))      # fp64 truth of the same algebra
        relmax = lambda a, b: float(np.max(np.abs(np.asarray(a, np.float64) - b)) / max(np.max(np.abs(b)), 1e-30))
        mine = {"idx_equal": bool(np.array_equal(o[4].cpu().numpy().reshape(-1), t.idx)),
                "classes": relmax(o[0].cpu().numpy(), t.classes[lo:hi]), "A": relmax(o[2].cpu().numpy(), t.A[lo:hi]),
                "B": relmax(o[3].cpu().numpy().reshape(C, D), np.asarray(t.B).reshape(C, D)), "pred_abs": float(np.max(np.abs(o[1].cpu().numpy().reshape(-1) - t.prediction_bag.reshape(-1))))}
        ok = mine["idx_equal"] and mine["classes"] < 2e-6 and mine["A"] < 2e-5 and mine["B"] < 1e-5
        flag = torch.tensor([1.0 if ok else 0.0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        parity = dict(mine, ok_all_ranks=bool(flag.item() == 1.0), N=Nc,
                      checker="oracle/dsmil_oracle.py forward() on the full bag (fp32 restatement of dsmil.py:46-62)")

    cpu_baseline = None
    extras = None
    if rank == 0 and world == 1:
        rate, arm, nrun = cpu_port_rate(p, args.cpu_seconds)
        cpu_baseline = {"value": rate, "unit": "patches/s", "cores": arm.threads, "kind": arm.kind,
                        "sample": f"{nrun} forwards over 16 distinct N={NBAG} bags in ~{args.cpu_seconds:.0f}s; {arm.what}"}
        if not args.no_extras:
            extras = run_extras(args, p, net, bags, dev, ms_per_step)
    if rank == 0:
        out = {"metric": METRIC, "value": value, "unit": "patches/s", "n_gpus": world, "steps": args.steps,
               "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "slides_per_sec": value / (NBAG * world),
               "config": {"workload": f"stream of {nb} synthetic bags per step, each N={NBAG * world} x D={D} fp32 "
                                      f"(U[0,1)), C={C}, nonlinear q, identity v; MILNet forward; "
                                      f"{'one GPU' if world == 1 else f'rows sharded over {world} GPUs ({NBAG} rows/rank/bag)'}",
                          "bags_per_step": nb, "rows_per_rank_per_bag": NBAG, "parallelism": f"row-shard x{world}",
                          "step_launch": graph_note if world > 1 else "eager: one forward_bags call per step",
                          "l2_policy": f"inputs larger than L2: {nb} bags x {NBAG * D * 4 / 1e6:.1f} MB per rank cycled",
                          "forward_path": int(lib.dsmil_forward_path(ctypes.byref(_lib.DsmilParams(D, C, 1, 0)), NBAG))},
               "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": launches * world,
               "clocks": clocks, "strong_n100k": strong, "parity_check": parity, "step_breakdown": breakdown,
               "embed_aggregate_resnet18": embed_agg, "extras": extras}
        print(json.dumps(out))
    if world > 1:
        # CUDA graphs that captured NCCL collectives keep communicator resources alive; tearing the process group down
        # underneath them can block forever (seen once: the JSON line was out, the process never exited).  Drop the
        # graphs, meet at a barrier, flush, and leave without running destructors.
        plan = None
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--bags", type=int, default=16, help="bags per step (16 x 20.5 MB > L2)")
    ap.add_argument("--ref-bags", type=int, default=16)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-graph", action="store_true", help="multi-GPU: host-launched step instead of the CUDA-graph replay")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra workloads (eager-GPU baseline, N=8192, "
                    "N=15000 training step, N=100k strong scaling, multi-rank parity check)")
    ap.add_argument("--giant-bags", type=int, default=32, help="N=100 000 bags per step of the strong-scaling workload")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy "
                    "(inputs are seeded: two builds run with the same arguments can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1 or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs needs --impl ours on one GPU")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
