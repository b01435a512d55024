#!/usr/bin/env python
"""bench.py — throughput of the HR-VITON hot path on B200 (driver contract: see the task statement).

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference algorithm on the host CPU cores (oracle port)
    python bench.py --dump-outputs DIR ...    # also write what the last timed step computed, DIR/<name>.npy

Prints ONE JSON line on rank 0.  Workloads (config.workload):
  train_stage2  (default) one full train_generator.py step per "step": frozen tocg -> warp -> SPADE G fwd+bwd -> D fwd+bwd
                (hinge + feature matching) + VGG loss -> Adam(G), then the D update (2nd G fwd, D fwd+bwd, Adam(D)),
                1024x768, bf16 activations (BASELINE.json configs[3], per-GPU batch --batch)
  train_stage1  one full train_condition.py step (tocg fwd+bwd with train-mode BatchNorm, stage-1 D, L1+VGG+TV+CE+LSGAN, Adam x2),
                1024x768 per-GPU batch 4 (BASELINE.json configs[1])
  gen_fwd       SPADEGenerator inference forward, 1024x768, per-GPU batch 8 (BASELINE.json configs[2])
  pipeline      end-to-end test_generator.py inference (tocg -> glue -> SPADE G), 1024x768, per-GPU batch 16 (BASELINE.json configs[4])
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # a benchmark run leaves the tree as it found it (it may be read-only)

H, W = 1024, 768
GEN_GFLOP_PER_IMG = 1636.4  # SURVEY.md §8(d): conv FLOPs of one SPADEGenerator forward at 1024x768


def gen_opt():
    return types.SimpleNamespace(norm_G="spectralaliasinstance", gen_semantic_nc=7, ngf=64, num_upsampling_layers="most",
                                 fine_height=H, fine_width=W, cuda=True)


TRAIN_STAGE2_WORKLOAD = ("train_stage2: full train_generator.py step (tocg fwd, G fwd+bwd, D fwd+bwd x2, 2nd G fwd, VGG loss fwd+dgrad, "
                         "Adam x2), 1024x768")


def conv_traffic():
    """Average DRAM bytes (read+write) per conv_igemm launch of one step, from the committed ncu pass
    (profiles/r2_conv_dram_traffic.json, written by tools/summarise_ncu_traffic.py from the ncu launch list of one step of the default
    command); None when that pass was not taken."""
    p = os.path.join(ROOT, "profiles", "r2_conv_dram_traffic.json")
    try:
        with open(p) as f:
            return json.load(f)["avg_dram_bytes_per_launch"]
    except Exception:
        return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"], "src": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BYTES = 60 << 20  # --dump-outputs: all arrays together stay below 64 MB


def dump_outputs(out_dir, arrays):
    """Writes {name: tensor} as out_dir/<name>.npy, float64 kept and everything else as float32.  An array larger than its share of
    DUMP_BYTES is written as a fixed sample of its flattened elements (distinct positions drawn from a generator with a constant seed,
    so the same for the same size): two runs or two builds with the same arguments compare element for element."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // max(1, len(arrays))
    for name, t in arrays.items():
        t = torch.as_tensor(t).detach()
        t = t if t.dtype == torch.float64 else t.float()
        k = share // t.element_size()
        if t.numel() > k:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:k].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def build_generator(device):
    import torch

    import network_generator
    from hrviton_b200 import spade
    torch.manual_seed(0)
    g = network_generator.SPADEGenerator(gen_opt(), 9)
    g.init_weights("xavier", 0.02)
    with torch.no_grad():
        for m in g.modules():
            if isinstance(m, spade.SPADENorm):
                m.noise_scale.normal_(0.0, 0.1)
    g = g.to(device).eval()
    with torch.no_grad():  # realistic spectral-norm u/v (a fresh module holds random vectors)
        for m in g.modules():
            if hasattr(m, "weight_orig"):
                for _ in range(3):
                    spade._sigma(m, True)
    return g


def synth_batch(b, device, seed):
    import torch
    gen = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.rand((b, 9, H, W), generator=gen) * 2 - 1
    lab = torch.randint(0, 7, (b, H // 16, W // 16), generator=gen)
    lab = lab.repeat_interleave(16, 1).repeat_interleave(16, 2)
    seg = torch.zeros((b, 7, H, W)).scatter_(1, lab[:, None], 1.0)
    return x, seg


def cpu_baseline_gen(steps=1, warmup=0, budget_s=240.0):
    """The reference algorithm on the host cores: the oracle port (oracle/hrviton_oracle.py — the reference is Python and
    cannot travel to the GPU box, SURVEY.md §8c) — SPADEGenerator forward, fp32, one 1024x768 image per step."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import hrviton_oracle as orc
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    import network_generator
    torch.manual_seed(0)
    m = network_generator.SPADEGenerator(gen_opt(), 9)
    m.init_weights("xavier", 0.02)
    sd = {k: v.detach() for k, v in m.state_dict().items()}
    x, seg = synth_batch(1, "cpu", 1)
    noise_fn = lambda b, hh, ww: torch.randn(b, hh, ww)
    times = []
    t_begin = time.time()
    done = 0
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.time()
            orc.spade_generator_forward(sd, x, seg, noise_fn)
            dt = time.time() - t0
            if i >= warmup:
                times.append(dt)
                done += 1
            if time.time() - t_begin + dt > budget_s and done >= 1:
                break
    times.sort()
    med = times[len(times) // 2]
    return {"value": 1.0 / med, "unit": "images/s", "cores": cores, "kind": "port",
            "sample": "SPADEGenerator fwd fp32, 1 image 1024x768 per step, %d timed step(s), torch %s CPU" % (len(times), torch.__version__),
            "s_per_image": med, "steps_done": len(times)}


def _reference_modules():
    """(networks, network_generator) of the UNMODIFIED reference (hrv_env.reference_dir(): the modules build() compiled into
    oracle/_ref, or a checkout named by $HRV_REFERENCE_DIR), imported under private names so that they cannot be confused with this
    repo's drop-ins of the same file names.  None when neither exists."""
    import importlib.util

    import hrv_env
    d = hrv_env.reference_dir()
    if d is None or not all(hrv_env.reference_file(d, n) for n in ("networks", "network_generator")):
        return None
    mods = []
    for name in ("networks", "network_generator"):
        spec = importlib.util.spec_from_file_location("hrv_reference_" + name, hrv_env.reference_file(d, name))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        mods.append(m)
    return mods[0], mods[1], d


def reference_stage2_step(nets, opts, batch, h, w, opt_g, opt_d):
    """One train_generator.py step (train_generator.py:201-360; opt.GT False, --occlusion off, clothmask_composition 'warp_grad') written
    against plain torch modules — used ONLY for the baseline arms (`--impl reference`: the reference's modules on the host CPU;
    `--impl torch_gpu`: the same modules on the GPU = PyTorch eager / cuDNN).  None of this repo's kernels is on this path."""
    import torch
    import torch.nn.functional as F
    from hrviton_b200 import train_step  # only the pure-torch helpers below (gaussian_blur_15_3, LABELS7): no kernel is touched
    tocg, G, D, vgg = nets
    dev = batch["cloth"].device
    cm, c_paired, im = batch["cloth_mask"], batch["cloth"], batch["image"]
    with torch.no_grad():
        input1 = torch.cat([F.interpolate(c_paired, size=(256, 192), mode="bilinear"), F.interpolate(cm, size=(256, 192), mode="nearest")], 1)
        input2 = torch.cat([F.interpolate(batch["parse_agnostic"], size=(256, 192), mode="nearest"),
                            F.interpolate(batch["densepose"], size=(256, 192), mode="bilinear")], 1)
        flow_list, fake_segmap, _, warped_cm = tocg(opts["tocg"], input1, input2)
        mask = torch.ones_like(fake_segmap)
        mask[:, 3:4] = warped_cm
        fake_segmap = fake_segmap * mask
        n = c_paired.shape[0]
        gx = torch.linspace(-1.0, 1.0, w, device=dev).view(1, 1, w, 1).expand(n, h, -1, -1)
        gy = torch.linspace(-1.0, 1.0, h, device=dev).view(1, h, 1, 1).expand(n, -1, w, -1)
        flow = F.interpolate(flow_list[-1].permute(0, 3, 1, 2), size=(h, w), mode="bilinear").permute(0, 2, 3, 1)
        grid = torch.cat([gx, gy], 3) + torch.cat([flow[..., 0:1] / ((96 - 1.0) / 2.0), flow[..., 1:2] / ((128 - 1.0) / 2.0)], 3)
        warped_cloth = F.grid_sample(c_paired, grid, padding_mode="border", align_corners=False)
        gauss = train_step.gaussian_blur_15_3(F.interpolate(fake_segmap, size=(h, w), mode="bilinear"))
        old_parse = torch.zeros(n, 13, h, w, device=dev).scatter_(1, gauss.argmax(dim=1)[:, None], 1.0)
        parse = torch.stack([old_parse[:, idx].sum(1) for idx in train_step.LABELS7], 1)
        g_in = torch.cat((batch["agnostic"], batch["densepose"], warped_cloth), 1)
    hinge_g = lambda preds: sum(-p[-1].mean() for p in preds) / len(preds)

    def hinge_d(preds, real):
        return sum(-torch.mean(torch.clamp((p[-1] - 1) if real else (-p[-1] - 1), max=0.0)) for p in preds) / len(preds)

    out = G(g_in, parse)
    pred = D(torch.cat((torch.cat((parse, out), 1), torch.cat((parse, im), 1)), 0))
    fake = [[t[:t.size(0) // 2] for t in p] for p in pred]
    real = [[t[t.size(0) // 2:] for t in p] for p in pred]
    loss_feat = sum(F.l1_loss(fake[i][j], real[i][j].detach()) * 10.0 / len(fake) for i in range(len(fake)) for j in range(len(fake[i]) - 1))
    fx, fy = vgg(out), vgg(im)
    loss_vgg = sum(wt * F.l1_loss(a, b.detach()) for wt, a, b in zip([1.0 / 32, 1.0 / 16, 1.0 / 8, 1.0 / 4, 1.0], fx, fy)) * 10.0
    loss_gen = hinge_g(fake) + loss_feat + loss_vgg
    opt_g.zero_grad()
    loss_gen.backward()
    opt_g.step()
    with torch.no_grad():
        out2 = G(g_in, parse)
    pred = D(torch.cat((torch.cat((parse, out2), 1), torch.cat((parse, im), 1)), 0))
    fake = [[t[:t.size(0) // 2] for t in p] for p in pred]
    real = [[t[t.size(0) // 2:] for t in p] for p in pred]
    loss_dis = hinge_d(fake, False) + hinge_d(real, True)
    opt_d.zero_grad()
    loss_dis.backward()
    opt_d.step()
    return float(loss_gen), float(loss_dis)


def build_reference_nets(ref, h, w, device):
    import torch
    rn, rg, _ = ref
    torch.manual_seed(0)
    topt = types.SimpleNamespace(warp_feature="T1", out_layer="relu", cuda=(device != "cpu"))
    tocg = rn.ConditionGenerator(topt, 4, 16, 13, ngf=96, norm_layer=torch.nn.BatchNorm2d).to(device).eval()
    gopt = gen_opt()
    gopt.fine_height, gopt.fine_width = h, w
    gopt.cuda = device != "cpu"  # SPADENorm draws its noise on opt.cuda's device (network_generator.py:104-107)
    gopt.ndf, gopt.norm_D, gopt.n_layers_D, gopt.num_D, gopt.no_ganFeat_loss = 64, "spectralinstance", 3, 2, False
    G = rg.SPADEGenerator(gopt, 9)
    G.init_weights("xavier", 0.02)
    D = rg.MultiscaleDiscriminator(gopt)
    D.init_weights("xavier", 0.02)
    G, D = G.to(device).train(), D.to(device).train()
    from torchvision import models
    feats = models.vgg19(weights=None).features  # random init: the pretrained file cannot be downloaded here (same as our arm)

    class Vgg(torch.nn.Module):  # networks.Vgg19 of the reference downloads weights in its constructor; same slicing (networks.py:201-231)
        def __init__(self):
            super().__init__()
            cuts = [0, 2, 7, 12, 21, 30]
            self.slices = torch.nn.ModuleList([torch.nn.Sequential(*[feats[i] for i in range(cuts[k], cuts[k + 1])]) for k in range(5)])
            for p in self.parameters():
                p.requires_grad = False

        def forward(self, x):
            out = []
            for sl in self.slices:
                x = sl(x)
                out.append(x)
            return out
    vgg = Vgg().to(device).eval()
    opt_g = torch.optim.Adam(G.parameters(), lr=1e-4, betas=(0.0, 0.9))
    opt_d = torch.optim.Adam(D.parameters(), lr=4e-4, betas=(0.0, 0.9))
    return (tocg, G, D, vgg), {"tocg": topt}, opt_g, opt_d


def host_threads():
    """Threads the CPU arm should use: the cores this process may actually run on — scheduler affinity, the cgroup CPU quota and
    the number of PHYSICAL cores behind the affinity mask, whichever is smallest.  (Round 2, first try: os.cpu_count() = 128 hardware
    threads on the GPU box made one reference step take 139 s — slower than the same step on 8 cores of the build container, 31 s:
    oversubscribed OpenMP teams.)"""
    try:
        aff = sorted(os.sched_getaffinity(0))
    except AttributeError:
        aff = list(range(os.cpu_count() or 1))
    n = len(aff)
    try:  # cgroup v2 quota
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    try:  # physical cores among the allowed logical CPUs
        cores, cur = set(), {}
        for ln in open("/proc/cpuinfo"):
            if ":" in ln:
                k, v = [t.strip() for t in ln.split(":", 1)]
                cur[k] = v
            elif cur:
                if int(cur.get("processor", -1)) in aff:
                    cores.add((cur.get("physical id", "0"), cur.get("core id", cur.get("processor"))))
                cur = {}
        if cores:
            n = min(n, len(cores))
    except Exception:
        pass
    env = os.environ.get("HRV_REF_THREADS")
    return max(1, int(env)) if env else max(1, n)


def cpu_baseline_train(steps=3, warmup=1, budget_s=200.0, size=(512, 384)):
    """The reference's own modules (oracle/_ref) running one REAL train_generator.py step per timed step on the host cores: tocg
    fwd (256x192, as in the reference) -> glue -> G fwd+bwd -> D -> hinge/feature-matching/VGG -> Adam(G) -> 2nd G fwd -> D fwd+bwd ->
    Adam(D), fp32, batch 1 at 512x384 — a quarter of the benchmarked pixel count and the smallest 4:3 size the reference generator
    admits (its latent grid is fine_width // 128 wide).  Reported as 1024x768-equivalent images/s (x 1/4: the three networks are fully
    convolutional, cost scales with pixels; the 256x192 tocg is NOT scaled down, which favours the CPU slightly).
    `warmup` / `steps` are honoured while the wall budget lasts: the loop stops early (never before one warm-up and one timed step)
    when the next step would overrun `budget_s`; what was actually run is returned and printed.  Falls back to the oracle port's
    generator fwd+bwd (kind 'port') only when the reference modules are absent."""
    import torch
    cores = host_threads()
    torch.set_num_threads(cores)
    ref = _reference_modules()
    if ref is None:
        return _cpu_baseline_port()
    import hrv_loader
    hrv_loader.load()
    from hrviton_b200 import train_step
    h, w = size
    nets, opts, opt_g, opt_d = build_reference_nets(ref, h, w, "cpu")
    batch = train_step.synthetic_batch(1, h, w, "cpu", seed=100)
    times, warm_done = [], 0
    t_begin = time.time()
    warmup = max(1, warmup)  # the first step pays oneDNN primitive creation (2-3x a steady step)
    while len(times) < steps:
        t0 = time.time()
        reference_stage2_step(nets, opts, batch, h, w, opt_g, opt_d)
        dt = time.time() - t0
        elapsed = time.time() - t_begin
        if warm_done < warmup:
            warm_done += 1
            if (budget_s - elapsed) < (warmup - warm_done + steps) * dt * 0.6:
                warmup = warm_done  # budget: spend what is left on timed steps, not on more warm-ups
            continue
        times.append(dt)
        if elapsed + dt > budget_s:
            break
    mean = sum(times) / len(times)
    scale = (h * w) / float(H * W)
    return {"value": scale / mean, "unit": "images/s", "cores": cores, "kind": "reference",
            "sample": "UNMODIFIED reference modules (%s), one full train_generator.py step per timed step, fp32, batch 1 at %dx%d (%.3g of the 1024x768 pixels; value = %.3g / step seconds), %d warm-up + %d timed steps, mean %.2f s/step, torch %s CPU, %d threads"
                      % (os.path.relpath(ref[2], ROOT) if ref[2].startswith(ROOT) else ref[2], h, w, scale, scale, warm_done, len(times), mean, torch.__version__, cores),
            "s_per_step": mean, "steps_done": len(times), "warmup_done": warm_done, "pixel_scale": scale}


def _cpu_baseline_port():
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import hrviton_oracle as orc
    cores = os.cpu_count() or 1
    import network_generator
    torch.manual_seed(0)
    opt = gen_opt()
    opt.fine_height, opt.fine_width = 512, 384
    m = network_generator.SPADEGenerator(opt, 9)
    m.init_weights("xavier", 0.02)
    sd = {k: v.detach().clone().requires_grad_(v.is_floating_point() and not k.endswith(("weight_u", "weight_v"))) for k, v in m.state_dict().items()}
    x = torch.rand(1, 9, 512, 384) * 2 - 1
    seg = torch.zeros(1, 7, 512, 384)
    seg[:, 0] = 1
    t0 = time.time()
    out = orc.spade_generator_forward(sd, x, seg, lambda b, hh, ww: torch.randn(b, hh, ww))
    out.mean().backward()
    dt = time.time() - t0
    return {"value": 0.25 / dt, "unit": "images/s", "cores": cores, "kind": "port",
            "sample": "NO reference modules (oracle/_ref): oracle port, SPADEGenerator fwd+bwd only on one 512x384 image (%.1f s), x1/4 pixel scaling" % dt,
            "s_per_step": dt, "steps_done": 1, "warmup_done": 0, "pixel_scale": 0.25}


def run_reference(args):
    """The driver's reference arm: the UNMODIFIED reference modules on the host cores (module docstring, cpu_baseline_train).  One
    timed step = one real train_generator.py step on a bounded sample (batch 1 at 512x384 = 0.25 image-equivalents of 1024x768);
    `ms_per_step` is the MEASURED wall time of such a step, `value` = 0.25 / that.  --steps / --warmup are honoured up to a wall
    budget (--ref-budget-s, default 240 s) so the arm ends within a few minutes whatever the box's cores; `steps` / `warmup` in the
    line are what actually ran (the requests are kept beside them)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    budget = float(os.environ.get("HRV_REF_BUDGET_S", "240"))
    if args.workload in ("train_stage2", "pipeline"):
        cb = cpu_baseline_train(steps=max(1, args.steps), warmup=max(1, args.warmup), budget_s=budget)
        wl = TRAIN_STAGE2_WORKLOAD
        ms = cb["s_per_step"] * 1e3
        per_step = cb["pixel_scale"]
    else:
        cb = cpu_baseline_gen(steps=max(1, args.steps), warmup=min(args.warmup, 1))
        cb["warmup_done"] = min(args.warmup, 1)
        wl = "gen_fwd: SPADEGenerator inference forward, 1024x768, bf16 activations, fp32 accumulate"
        ms = cb["s_per_image"] * 1e3
        per_step = 1.0
    line = {"impl": "reference", "metric": "1024x768 try-on images/sec", "value": cb["value"], "unit": "images/s", "n_gpus": args.gpus,
            "steps": cb["steps_done"], "warmup": cb["warmup_done"], "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl, "launch": "eager, host CPU (%d threads)" % cb["cores"], "feeding": "host tensors",
                       "per_gpu_batch": 8, "global_batch": 8, "parallelism": "dp1",
                       "sample": cb["sample"], "images_per_step": per_step,
                       "steps_requested": args.steps, "warmup_requested": args.warmup, "wall_budget_s": budget},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_torch_gpu(args):
    """Context line (not a driver arm): the reference's modules themselves on the GPU — PyTorch eager / cuDNN, fp32 (TF32 convolutions
    as torch defaults) or bf16 autocast — one full train_generator.py step at 1024x768.  SURVEY.md §2 names this as the real bar."""
    import torch
    ref = _reference_modules()
    if ref is None:
        print(json.dumps({"impl": "torch_gpu", "unavailable": "no reference modules (oracle/_ref)"}))
        return
    import hrv_loader
    hrv_loader.load()
    from hrviton_b200 import train_step
    dev = "cuda"
    B = args.batch or 2
    nets, opts, opt_g, opt_d = build_reference_nets(ref, H, W, dev)
    batch = train_step.synthetic_batch(B, H, W, dev, seed=100)
    amp = os.environ.get("HRV_TORCH_GPU_AMP", "bf16")
    ctx = (lambda: torch.autocast("cuda", dtype=torch.bfloat16)) if amp == "bf16" else (lambda: torch.autocast("cuda", enabled=False))
    torch.backends.cudnn.benchmark = True

    def step():
        with ctx():
            return reference_stage2_step(nets, opts, batch, H, W, opt_g, opt_d)
    for _ in range(max(2, args.warmup)):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    print(json.dumps({"impl": "torch_gpu", "metric": "1024x768 try-on images/sec", "value": B / (ms / 1e3), "unit": "images/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": max(2, args.warmup), "ms_per_step": ms, "dtype": amp, "data": "synthetic",
                      "config": {"workload": "train_stage2: full train_generator.py step, UNMODIFIED reference modules on the GPU (PyTorch %s eager, cuDNN, autocast %s), 1024x768" % (torch.__version__, amp),
                                 "per_gpu_batch": B, "peak_mem_GB": torch.cuda.max_memory_allocated() / 1e9}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_gpu"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: 8 for train_stage2 and gen_fwd, 4 for train_stage1)")
    ap.add_argument("--workload", default="train_stage2", choices=["train_stage2", "train_stage1", "gen_fwd", "pipeline"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="train_stage2: launch eagerly instead of replaying a CUDA graph")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: per-GPU batch fixed (default 8); strong: GLOBAL batch fixed at --batch (default 8), split over the ranks")
    ap.add_argument("--dump-profile", default="", help="write the per-launch CUDA-event profile of one step as CSV")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (training: its losses and the updated parameters)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "torch_gpu":
        return run_torch_gpu(args)

    # NCCL prints its version banner on STDOUT at NCCL_DEBUG=VERSION (the image's default): keep stdout to the one JSON line
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"
    import torch
    import torch.distributed as dist

    import hrv_loader
    hrv_loader.load()
    from hrviton_b200 import ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W_ = max(3, args.warmup)
    K = args.steps
    train = args.workload in ("train_stage2", "train_stage1")
    stage1 = args.workload == "train_stage1"
    pipe = args.workload == "pipeline"
    B = args.batch or (4 if stage1 else (16 if pipe else 8))
    if args.scaling == "strong":
        if B % world:
            raise SystemExit("--scaling strong: global batch %d is not divisible by %d ranks" % (B, world))
        B = B // world

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if train:
        os.environ.setdefault("HRV_VGG_RANDOM_INIT", "1")  # no network: torchvision weights cannot be downloaded
        import network_generator
        import networks
        from hrviton_b200 import ddp, train_step
        topt = types.SimpleNamespace(warp_feature="T1", out_layer="relu", cuda=True)
        torch.manual_seed(0)
        tocg = networks.ConditionGenerator(topt, 4, 16, 13, ngf=96, norm_layer=torch.nn.BatchNorm2d)
        with torch.no_grad():
            for mod in tocg.modules():
                if isinstance(mod, torch.nn.BatchNorm2d):
                    mod.running_mean.normal_(0, 0.1)
                    mod.running_var.uniform_(0.5, 1.5)
        tocg = tocg.to(dev).eval()
        g = None if stage1 else build_generator(dev).train()
        dopt = gen_opt()
        dopt.ndf, dopt.norm_D, dopt.n_layers_D, dopt.num_D, dopt.no_ganFeat_loss = 64, "spectralinstance", 3, 2, False
        vgg = networks.Vgg19().to(dev).eval()
        reducers = {}
        if stage1:
            import contextlib
            import io
            tocg.train()
            with contextlib.redirect_stdout(io.StringIO()):
                D = networks.define_D(input_nc=33, Ddownx2=True, Ddropout=True, n_layers_D=3, spectral=False, num_D=2)
            D = D.to(dev).train()
            if world > 1:
                reducers = {"G": ddp.GradBucketReducer(list(tocg.parameters())), "D": ddp.GradBucketReducer(list(D.parameters()))}
            tr1 = train_step.Stage1Trainer(tocg, D, vgg, reducers=reducers)

            class _Shim:  # same step/capture/replay surface as Stage2Trainer
                def step(self, b, h, w):
                    return tr1.step(b)

                def capture(self, b, h, w):
                    tr1.capture(b)

                def replay(self, b=None, feeder=None):
                    return tr1.replay(b, feeder=feeder)
            trainer = _Shim()
            make_batch = train_step.synthetic_batch_stage1
        else:
            D = network_generator.MultiscaleDiscriminator(dopt)
            D.init_weights("xavier", 0.02)
            D = D.to(dev).train()
            if world > 1:
                reducers = {"G": ddp.GradBucketReducer(list(g.parameters())), "D": ddp.GradBucketReducer(list(D.parameters()))}
            trainer = train_step.Stage2Trainer(tocg, g, D, vgg, reducers=reducers)
            make_batch = train_step.synthetic_batch
        batch_cpu = make_batch(B, H, W, "cpu", seed=100 + rank)
        batch_d = {k: v.to(dev) for k, v in batch_cpu.items()}
        feeder = train_step.BatchFeeder(batch_cpu, dev)  # pinned host copies; one-hot maps as uint8 labels; double-buffered copy stream
        del batch_cpu
        loss_h = torch.empty(2, dtype=torch.float32).pin_memory()
        h2d_bytes = feeder.bytes_per_step
        d2h_bytes = 8

        # One CUDA graph per step.  With more than one rank the NCCL bucket all-reduces (launched from gradient hooks during
        # backward) are captured into the same graph; HRV_MULTI_GRAPH=0 forces eager launches for N > 1.
        use_graph = not args.no_graph and (world == 1 or os.environ.get("HRV_MULTI_GRAPH", "1") != "0")
        if use_graph:
            try:
                for _ in range(2 if world > 1 else 1):
                    trainer.step(batch_d, H, W)  # eager steps first: lazy initialisation (optimizer state, caches, NCCL communicator, gradient buckets)
                barrier()
                l_cap = ops.LAUNCHES[0]
                trainer.capture(batch_d, H, W)
                launches_per_replay = (ops.LAUNCHES[0] - l_cap) // 3  # capture() runs 2 warm steps + the captured one
            except Exception as e:  # noqa: BLE001 - report and fall back to eager launches
                import traceback
                sys.stderr.write("CUDA graph capture failed (%s: %s); running eagerly\n%s\n" % (type(e).__name__, e, traceback.format_exc()[-1500:]))
                use_graph = False
        if world > 1:  # every rank must take the same path
            flag = torch.tensor([1 if use_graph else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if use_graph and not int(flag.item()):
                raise SystemExit("graph capture succeeded on this rank but failed on another: rerun with HRV_MULTI_GRAPH=0")

        def step_resident():
            if use_graph:
                ops.LAUNCHES[0] += launches_per_replay
                return trainer.replay()
            return trainer.step(batch_d, H, W)

        feeder.prefetch()  # the first batch of the e2e loop is in flight before its first step (every later one overlaps a step)

        def step_e2e():
            if use_graph:
                ops.LAUNCHES[0] += launches_per_replay + len(feeder.classes)
                out = trainer.replay(feeder=feeder)
            else:
                out = trainer.step(feeder.consume(batch_d), H, W)
            lk = ("loss_g", "loss_d") if stage1 else ("loss_gen", "loss_dis")
            loss_h.copy_(torch.stack([out[lk[0]].float(), out[lk[1]].float()]), non_blocking=True)
    elif pipe:
        # BASELINE.json configs[4]: the end-to-end test_generator.py pipeline (tocg -> parse post-processing -> hi-res warp with occlusion
        # handling -> SPADEGenerator), 1024x768, batch 16, inference
        import networks
        from hrviton_b200 import pipeline, train_step
        topt = types.SimpleNamespace(warp_feature="T1", out_layer="relu", cuda=True)
        torch.manual_seed(0)
        tocg = networks.ConditionGenerator(topt, 4, 16, 13, ngf=96, norm_layer=torch.nn.BatchNorm2d)
        with torch.no_grad():
            for mod in tocg.modules():
                if isinstance(mod, torch.nn.BatchNorm2d):
                    mod.running_mean.normal_(0, 0.1)
                    mod.running_var.uniform_(0.5, 1.5)
        tocg = tocg.to(dev).eval()
        g = build_generator(dev)
        batch_cpu = train_step.synthetic_batch(B, H, W, "cpu", seed=100 + rank)
        batch_d = {k: v.to(dev) for k, v in batch_cpu.items()}
        feeder = train_step.BatchFeeder(batch_cpu, dev)
        del batch_cpu
        out_h = torch.empty((B, 3, H, W), dtype=torch.float32).pin_memory()
        h2d_bytes = feeder.bytes_per_step
        d2h_bytes = int(out_h.numel() * 4)

        def step_resident():
            return pipeline.tryon_forward(tocg, g, batch_d, occlusion=True)[0]

        feeder.prefetch()

        def step_e2e():
            out = pipeline.tryon_forward(tocg, g, feeder.consume(batch_d), occlusion=True)[0]
            out_h.copy_(out, non_blocking=True)
    else:
        g = build_generator(dev)
        x_h, seg_h = synth_batch(B, "cpu", 100 + rank)
        x_h, seg_h = x_h.pin_memory(), seg_h.pin_memory()
        x_d, seg_d = x_h.to(dev), seg_h.to(dev)
        out_h = torch.empty((B, 3, H, W), dtype=torch.float32).pin_memory()
        h2d_bytes = int(x_h.numel() * 4 + seg_h.numel() * 4)
        d2h_bytes = int(out_h.numel() * 4)

        def step_resident():
            with torch.no_grad():
                return g(x_d, seg_d)

        def step_e2e():
            with torch.no_grad():
                xd = x_h.to(dev, non_blocking=True)
                sd = seg_h.to(dev, non_blocking=True)
                out = g(xd, sd)
                out_h.copy_(out, non_blocking=True)

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            out = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, out

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # started before the warm-up: nvidia-smi needs ~0.5 s to emit its first sample
    for _ in range(W_):
        step_resident()
    if rank == 0:
        sampler.lines.clear()  # keep only samples taken during the timed region
    l0 = ops.LAUNCHES[0]
    ms, out = timed(step_resident, K)
    launches = ops.LAUNCHES[0] - l0
    clocks = sampler.stop() if rank == 0 else None
    value = B * world * K / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        # before anything else runs: the steps below keep training the same parameters and reuse the graph's output buffers
        arrays = dict(out) if isinstance(out, dict) else {"output": out}
        if train:
            for tag, net in ((("tocg", tocg) if stage1 else ("generator", g)), ("discriminator", D)):
                arrays[tag + "_params"] = torch.cat([p.detach().reshape(-1).float() for p in net.parameters()])
        dump_outputs(args.dump_outputs, arrays)

    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, K)
    e2e_value = B * world * K / (ms_e2e / 1e3)

    # ---- per-kernel profile pass (CUDA events around every C-ABI launch) -> roofline of the dominant kernel
    ops.PROFILE = []
    torch.cuda.synchronize()
    # process-wide start/end range (the backward runs on autograd's own thread, which a push/pop range would not cover):
    # `ncu --nvtx --nvtx-include "hrv_profile_step" ...` = launch list of exactly ONE step of this command
    nvtx_id = torch.cuda.nvtx.range_start("hrv_profile_step")
    if train:
        trainer.step(batch_d, H, W)  # eager (events cannot be recorded inside a graph replay)
    else:
        step_resident()
    torch.cuda.synchronize()
    torch.cuda.nvtx.range_end(nvtx_id)
    prof = ops.PROFILE
    ops.PROFILE = None
    agg = {}
    if args.dump_profile and rank == 0:
        with open(args.dump_profile, "w") as f:
            f.write("kind,label,ms,work,rate_T_per_s\n")
            for kind, work, e0, e1, label in prof:
                t = e0.elapsed_time(e1)
                f.write("%s,%s,%.4f,%.4g,%.2f\n" % (kind, label, t, work, work / (t * 1e-3) / 1e12 if t > 0 else 0))
    for kind, work, e0, e1, _label in prof:
        a = agg.setdefault(kind, [0.0, 0.0, 0])
        a[0] += work
        a[1] += e0.elapsed_time(e1)
        a[2] += 1
    peaks = measured_peaks()
    conv_flops = agg.get("conv", [0, 0, 0])[0] + agg.get("conv_spade", [0, 0, 0])[0]
    conv_ms = agg.get("conv", [0, 0, 0])[1] + agg.get("conv_spade", [0, 0, 0])[1]
    conv_launches = agg.get("conv", [0, 0, 0])[2] + agg.get("conv_spade", [0, 0, 0])[2]
    achieved = conv_flops / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
    roofline = {"kernel": "conv_pair_kernel + conv_pixn_kernel + conv_igemm_kernel (tcgen05 implicit-GEMM convolution, all %d launches of one step)" % conv_launches,
                "bound": "tensor", "achieved": achieved, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                "frac": achieved / peaks["tf_sustained"],
                "traffic": conv_traffic() if (train and not stage1 and B == 8) else None,  # the ncu pass was taken on the default workload only
                "peak_source": peaks["src"] + " (bf16 sustained)",
                "avg_launch_ms": conv_ms / max(1, conv_launches), "algorithmic_gflop_per_launch": conv_flops / 1e9 / max(1, conv_launches)}
    # The convolution launches are not all tensor-bound: the thin-channel full-resolution layers (3->64, 9->16, 32->3, the 1x1 64->128
    # after im2col ...) move more bytes than the tensor pipe needs time for.  Second figure: every launch against ITS OWN bound,
    # max(flops / tensor peak, algorithmic bytes / HBM peak), summed over the step and divided by the measured time.
    import re
    floor_ms, n_hbm = 0.0, 0
    for kind, work, e0, e1, label in prof:
        if kind not in ("conv", "conv_spade"):
            continue
        m = re.match(r"\s*(\d+)->(\d+) k(\d+)x(\d+) n(\d+) (\d+)x(\d+)", label or "")
        if not m:
            continue
        cin, ng, _kh, _kw, nb, hh, ww = (int(v) for v in m.groups())
        byt = float(nb) * hh * ww * ((cin + ng) * 2 + (4 if kind == "conv_spade" else 0))  # input + output (SPADE: gamma|beta columns <-> x read + out write) [+ noise]
        t_t, t_h = work / (peaks["tf_sustained"] * 1e12) * 1e3, byt / (peaks["hbm_gbs"] * 1e9) * 1e3
        floor_ms += max(t_t, t_h)
        n_hbm += 1 if t_h > t_t else 0
    if conv_ms > 0:
        roofline["frac_vs_per_launch_bound"] = floor_ms / conv_ms
        roofline["hbm_bound_launches"] = n_hbm
    total_prof_ms = sum(a[1] for a in agg.values())
    breakdown = {k: {"ms": round(a[1], 3), "launches": a[2], "share": round(a[1] / total_prof_ms, 4)} for k, a in agg.items()}
    if "instnorm_stats" in agg:
        a = agg["instnorm_stats"]
        breakdown["instnorm_stats"]["achieved_GBps"] = round(a[0] / (a[1] * 1e-3) / 1e9, 1)
        breakdown["instnorm_stats"]["frac_of_hbm_peak"] = round(a[0] / (a[1] * 1e-3) / 1e9 / peaks["hbm_gbs"], 4)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_baseline_train(steps=2, warmup=1, budget_s=60.0) if train else cpu_baseline_gen(steps=1, warmup=0)
        cpu_baseline = {k: cpu_baseline[k] for k in ("value", "unit", "cores", "kind", "sample")}

    if rank == 0:
        line = {"metric": "1024x768 try-on images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": K, "warmup": W_,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic",
                "config": {"workload": ("train_stage1: full train_condition.py step (tocg fwd+bwd with train-mode BatchNorm, 3 stage-1 D passes fwd+bwd, VGG loss x5 fwd+dgrad, L1/TV/CE/LSGAN, Adam x2; README flags --Ddownx2 --Ddropout --lasttvonly --interflowloss --occlusion), 1024x768, bf16 activations / fp32 accumulate" if (train and stage1) else
                                        TRAIN_STAGE2_WORKLOAD
                                        if train else ("pipeline: end-to-end test_generator.py inference (tocg 256x192 -> parse post-processing -> hi-res cloth warp with occlusion handling -> SPADEGenerator), 1024x768, bf16 activations / fp32 accumulate"
                                                       if pipe else "gen_fwd: SPADEGenerator inference forward, 1024x768, bf16 activations, fp32 accumulate")),
                           "kernels": ("bf16 activations / fp32 accumulate; convs (fwd/dgrad/wgrad), norms, modulation, activations, pooling, weight packing, parse-map and warp glue, VGG L1 on this repo's kernels; hinge/feature-matching reductions, spectral-norm power iteration, Adam = torch"
                                       if (train and not stage1) else "this repo's kernels (see DESIGN.md)"),
                           "launch": (("cuda-graph replay of the whole step" + (" (NCCL bucket all-reduces captured in the graph)" if world > 1 else "")) if (train and use_graph) else "eager"),
                           "feeding": "e2e: pinned host batch -> device on a copy stream, double-buffered (overlaps the previous step); one-hot parse maps shipped as uint8 labels and expanded by hrv_onehot_u8" if train else "e2e: pinned host -> device on the compute stream", "per_gpu_batch": B, "global_batch": B * world, "parallelism": "dp%d" % world,
                           "l2": "activations per step (>10 GB) exceed the 126 MB L2; no explicit flush",
                           "weights": "xavier(0.02) random init, noise_scale~N(0,0.1)"},
                "e2e": {"value": e2e_value, "unit": "images/s", "ms_per_step": ms_e2e / K,
                        "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes},
                "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "kernel_breakdown": breakdown,
                "model_tflops": (None if stage1 else (8800.0 if train else (GEN_GFLOP_PER_IMG + 91.75 if pipe else GEN_GFLOP_PER_IMG)) * value / 1e3)}
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        print(json.dumps(line))
    if world > 1:
        # Tear-down.  The result is already on stdout; nothing below may keep the job alive.  Graph nodes reference the NCCL
        # communicator (round 2: both 2-GPU graph runs printed their line and then sat in destroy_process_group until `timeout`
        # killed them), so the graph goes first, and a watchdog ends the process if the communicator still refuses to die.
        sys.stdout.flush()
        wd = threading.Timer(45.0, lambda: os._exit(0))
        wd.daemon = True
        wd.start()
        torch.cuda.synchronize()
        barrier()
        if train and use_graph:
            trainer.release_graph()
        dist.destroy_process_group()
        wd.cancel()
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        os._exit(0)  # skip interpreter-exit destructors of NCCL-bearing objects (same hang, later)


if __name__ == "__main__":
    main()
