#!/usr/bin/env python
"""bench.py — headline benchmark of the NS2VC denoiser hot path (BASELINE.json metric).

metric: denoiser-steps/s = B x (UNet forwards) per second over full 50-NFE DPM-Solver++(2M)
sampling runs at [B=8, C=100, T=1024], prompt S=256 (BASELINE.json configs[1]).

A bench "step" = ONE complete 50-step sampling run of one batch of 8 utterances per GPU
(prepare_cond + 50 x (UNet forward + fused sampler step); multi-GPU: + one all-gather of the final
latents).  `value` times device-resident inputs; `e2e` times the public API
(ns2vc_b200.api.sample_latents) from pinned host tensors to a host result, copies inside the timed
region.  Weak scaling over GPUs (independent utterances per rank, SURVEY.md §8e).

--dump-outputs DIR writes the final latents of the last timed step of both paths, [world x B, 100, T]
float32: DIR/latents.npy (`value`'s path) and DIR/latents_e2e.npy (`e2e`'s path).  Weights and inputs
are seeded, so the same arguments give the same inputs on every run.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

B, T, S, NFE = 8, 1024, 256, 50
METRIC = "denoiser-steps/s"
UNIT = "denoiser-steps/s"
# SURVEY.md 8(d): algorithmic work of one sample-step, F(T,S) FLOPs (conv + linear + QK^T/PV + the step-invariant K/V projections,
# counted because the reference executes them every step), and the ideal-fusion byte count (3.20 GB per cfg2 step, fp32 I/O)
def survey_flops(Bn, Tn, Sn):
    return Bn * (31818240 * Tn + 4352 * Tn * Tn + 7296 * Sn * Tn + 4456448 * Sn)
SURVEY_BYTES_CFG2 = 3.20e9


def workload_cfg(n_gpus):
    return {"workload": f"cfg2: B={B}/GPU, C=100, T={T}, S={S}, {NFE}-step DPM-Solver++(2M) multistep time_uniform, x_start UNet1D (66.08M params)",
            "global_batch": B * n_gpus, "nfe": NFE, "parallelism": f"utterance-shard x{n_gpus} (one all-gather of latents)" if n_gpus > 1 else "single GPU",
            "l2_policy": "per-forward weight stream (264 MB packed bf16 hi/lo + 2.9 GB activations) exceeds the 126 MB L2; no explicit flush"}


def flops_per_forward(cfg, Bn, Tn, Sn, gemm_only=False):
    """Algorithmic FLOPs of one UNet forward (SURVEY.md Appendix E work model), from the layer plan."""
    from ns2vc_b200.arch import build_plan, level_lengths
    Tl = level_lengths(Tn, len(cfg.block_out_channels))
    gemm = 2 * Tn * cfg.in_channels * cfg.block_out_channels[0] * 3 + 2 * Tn * cfg.block_out_channels[0] * cfg.out_channels * 3
    attn = 0
    for op in build_plan(cfg):
        t = Tl[op.level]
        if op.kind == "resnet":
            gemm += 2 * t * (3 * op.cin * op.cout + 3 * op.cout ** 2 + (op.cin != op.cout) * op.cin * op.cout)
        elif op.kind == "xformer":
            c = op.cout
            gemm += 2 * t * c * c * (1 + 3 + 1 + 1 + 1 + 8 + 4 + 1)
            attn += 4 * t * t * c + 4 * t * Sn * c
        elif op.kind in ("down", "up"):
            gemm += 2 * t * op.cout ** 2 * 3
    return Bn * (gemm if gemm_only else gemm + attn), Bn * attn


def read_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured (MEASURED_PEAKS.json, sustained bf16)"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi sampler running during the timed region (recipe's clocks line)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for i, n in enumerate(names):
                    if "Active" in r[3 + i] and "Not" not in r[3 + i]:
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def host_inputs(seed):
    from ns2vc_b200.synth import make_inputs
    inp = make_inputs(B, T, S, seed=seed)
    return {k: (v.pin_memory() if torch.cuda.is_available() else v) for k, v in inp.items()}


def host_threads():
    """Threads this process may really use: CPU affinity capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(int(q) / int(per))))
    except Exception:
        pass
    return n


def best_thread_count():
    """PyTorch CPU kernels stop scaling (and can collapse) far below the core count of a big host:
    pick the fastest of a few thread counts on a small forward, so the CPU baseline is not sandbagged."""
    from ns2vc_b200.arch import ns2vc_denoiser_config
    from ns2vc_b200.synth import make_inputs, make_state_dict
    from oracle import unet_oracle
    cfg = ns2vc_denoiser_config()
    sd = make_state_dict(cfg, 0)
    inp = make_inputs(2, 256, 64, seed=0)
    t = torch.full((2,), 500.0)
    cap = host_threads()
    best, best_dt = 1, float("inf")
    for n in sorted({c for c in (8, 16, 32, 64, cap) if c <= cap} or {cap}):
        torch.set_num_threads(n)
        with torch.no_grad():
            unet_oracle.denoiser_forward(sd, cfg, inp["x"], inp["content"], inp["prompt"], inp["refer_lengths"], t)
            t0 = time.perf_counter()
            unet_oracle.denoiser_forward(sd, cfg, inp["x"], inp["content"], inp["prompt"], inp["refer_lengths"], t)
            dt = time.perf_counter() - t0
        if dt < best_dt:
            best, best_dt = n, dt
    return best


def cpu_oracle_rate(n_forwards, threads):
    """The reference's CPU path for one denoiser call at the cfg2 shape, timed on the host cores through
    the oracle port (bit-identical restatement of the reference's ATen call sequence)."""
    from ns2vc_b200.arch import ns2vc_denoiser_config
    from ns2vc_b200.synth import make_inputs, make_state_dict
    from oracle import unet_oracle
    torch.set_num_threads(threads)
    cfg = ns2vc_denoiser_config()
    sd = make_state_dict(cfg, 0)
    inp = make_inputs(B, T, S, seed=0)
    t = torch.full((B,), 500.0)
    with torch.no_grad():
        unet_oracle.denoiser_forward(sd, cfg, inp["x"], inp["content"], inp["prompt"], inp["refer_lengths"], t)   # warm-up
        t0 = time.perf_counter()
        for _ in range(n_forwards):
            unet_oracle.denoiser_forward(sd, cfg, inp["x"], inp["content"], inp["prompt"], inp["refer_lengths"], t)
        dt = time.perf_counter() - t0
    return B * n_forwards / dt, dt


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = best_thread_count()
    per_step = 2                                     # bounded sample: 2 of the 50 denoiser calls per "step"
    from ns2vc_b200.arch import ns2vc_denoiser_config
    from ns2vc_b200.synth import make_inputs, make_state_dict, linear_betas
    from oracle import unet_oracle, sampler_oracle
    torch.set_num_threads(threads)
    cfg = ns2vc_denoiser_config()
    sd = make_state_dict(cfg, 0)
    inp = make_inputs(B, T, S, seed=0)
    sch = sampler_oracle.OracleSchedule(linear_betas(1000))
    fn = lambda x, tt: unet_oracle.denoiser_forward(sd, cfg, x, inp["content"], inp["prompt"], inp["refer_lengths"], tt)
    ts = torch.linspace(1.0, 1e-3, NFE + 1)

    def step():
        x = inp["x"]
        with torch.no_grad():
            for k in range(per_step):               # model call + x0 round trip, as the sampler does per NFE
                x = sampler_oracle.x0_model(fn, sch, x, ts[k])
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    val = B * per_step * args.steps / dt
    # one COMPLETE 50-NFE DPM-Solver++(2M) run of the reference path (outside the timed steps): the whole-run rate
    t1 = time.perf_counter()
    with torch.no_grad():
        sampler_oracle.dpmpp_2m(fn, sch, inp["x"], NFE)
    full_dt = time.perf_counter() - t1
    sample = f"{per_step} of {NFE} denoiser calls (UNet forward + x0 round trip) per step at B={B},T={T},S={S}; reference CPU path via the oracle port (reference is pure PyTorch; /root/reference is absent on the GPU box)"
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                      "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_cfg(args.gpus),
                      "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                                       "full_run": {"value": B * NFE / full_dt, "unit": UNIT, "seconds": full_dt, "what": f"one complete {NFE}-NFE DPM-Solver++(2M) run at B={B},T={T},S={S}"}},
                      "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "gpu_launches": 0}))


PRE_CFG = {"phoneme_encoder": dict(in_channels=256, hidden_channels=256, out_channels=256, n_layers=6, p_dropout=0.2),
           "prompt_encoder": dict(in_channels=100, hidden_channels=256, out_channels=256, n_layers=6, p_dropout=0.2)}     # reference config.json:27-49


def pre_flops(Bn, Tn, Sn, H=256, L=6, k=9):
    """Algorithmic FLOPs of Pre_model.infer: per frame and layer QKV + out-proj + k-tap conv-FFN (C -> 4C) + FFN out, the
    attention products, and the two k=1 ConvLayers of each encoder."""
    per_layer = 2 * H * 3 * H + 2 * H * H + 2 * H * 4 * H * k + 2 * 4 * H * H
    enc = lambda n, cin: Bn * n * (L * per_layer + 2 * cin * H + 2 * H * H) + Bn * L * 4 * n * n * H
    return enc(Tn, 256) + enc(Sn, 100)


def bench_pre_model(unet, dev, hin, nfe, with_cpu):
    from ns2vc_b200 import api
    from ns2vc_b200.pre_model import Pre_model
    from ns2vc_b200.synth import make_pre_inputs, make_pre_state_dict
    pre = Pre_model(PRE_CFG)
    sd = make_pre_state_dict(PRE_CFG, 0)
    pre.load_state_dict(sd)
    pre = pre.to(dev).eval()
    pin = make_pre_inputs(B, T, S, seed=5)
    pin_h = {k: v.pin_memory() for k, v in pin.items()}
    data = (pin["c"].to(dev), pin["refer"].to(dev), None, None, None, pin["lengths"].to(dev), pin["refer_lengths"].to(dev), None)
    for _ in range(3):
        pre.infer(data)
    torch.cuda.synchronize(dev)
    K = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        pre.infer(data)
    e1.record(); torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / K
    fl = pre_flops(B, T, S)
    peaks = read_peaks()
    res = {"workload": f"Pre_model.infer (ref_enc + PromptEncoder + PhoneEncoder, 34.9M params) at B={B}, T={T}, S={S}, device-resident inputs",
           "ms_per_call": ms, "utterances_per_s": B / (ms / 1e3), "launches_per_call": pre.launch_count(), "algorithmic_gflop": fl / 1e9,
           "achieved_tflops": fl / (ms * 1e-3) / 1e12, "frac_of_tensor_peak": fl / (ms * 1e-3) / 1e12 / peaks["tflops"]}
    # whole device pipeline through the public API: host (pinned) features in, host latents out, copies inside the timed region
    def run():
        return api.sample_from_features(pre, unet, hin["x"], pin_h["c"], pin_h["refer"], pin_h["lengths"], pin_h["refer_lengths"], steps=nfe, device=dev).cpu()
    for _ in range(3):
        run()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(2):
        run()
    e1.record(); torch.cuda.synchronize(dev)
    mp = e0.elapsed_time(e1) / 2
    res["pipeline_e2e"] = {"what": f"api.sample_from_features: Pre_model.infer + {nfe}-NFE DPM-Solver++(2M) sampling, pinned host features in, host latents out",
                           "ms_per_run": mp, "value": B * nfe / (mp / 1e3), "unit": UNIT, "pre_model_share": ms / mp}
    if with_cpu:
        from oracle import pre_model_oracle as po                # CPU baseline leg: the oracle port of the reference's CPU path
        torch.set_num_threads(min(host_threads(), 32))
        with torch.no_grad():
            t0 = time.perf_counter()
            po.pre_model_infer(sd, pin["c"], pin["refer"], pin["lengths"], pin["refer_lengths"], 6, 6)
            dt = time.perf_counter() - t0
        res["cpu_baseline"] = {"ms_per_call": 1e3 * dt, "cores": torch.get_num_threads(), "kind": "port",
                               "sample": "one Pre_model.infer at the same shape through the oracle port of the reference's CPU PyTorch path"}
    del pre
    return res


def ncu_traffic(kernel):
    """Average DRAM bytes per launch of `kernel` from the committed ncu launch list (profiles/)."""
    p = os.path.join(REPO, "profiles", "r02_traffic.json")
    if not os.path.exists(p):
        p = os.path.join(REPO, "profiles", "r01_traffic.json")
    if not os.path.exists(p):
        return None
    tab = json.load(open(p))
    pref = "gemm_tc_kernel" if kernel == "gemm_tc" else "attn_v2_kernel"
    n = sum(v["launches"] for k, v in tab.items() if k.startswith(pref))
    tot = sum(v["launches"] * v["dram_bytes_per_launch"] for k, v in tab.items() if k.startswith(pref))
    return tot / n if n else None


DUMP_LIMIT_BYTES = 64 << 20


def write_dumps(path, arrays):
    """Write each tensor as float32 ``path/<name>.npy``; refuse rather than write more than DUMP_LIMIT_BYTES in all."""
    import numpy as np
    arrays = {k: v.detach().to("cpu", torch.float32).numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, f"{k}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--nfe", type=int, default=NFE, help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the latents of the last timed step as DIR/<name>.npy (float32) "
                         "so two builds can be compared output for output; the inputs are seeded")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the b200 path")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    assert args.warmup >= 3, "timing rules: W >= 3"
    import torch.distributed as dist
    from ns2vc_b200 import _lib, api
    from ns2vc_b200.arch import ns2vc_denoiser_config
    from ns2vc_b200.fused import DenoiserSession
    from ns2vc_b200.shard import gather_latents
    from ns2vc_b200.synth import make_state_dict
    from ns2vc_b200.unet import UNet1DConditionModel

    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    nfe = args.nfe
    cfg = ns2vc_denoiser_config()
    unet = UNet1DConditionModel(in_channels=356, out_channels=100, block_out_channels=(128, 256, 384, 512), norm_num_groups=8,
                                cross_attention_dim=256, attention_head_dim=8, addition_embed_type="text",
                                resnet_time_scale_shift="scale_shift")
    unet.load_state_dict(make_state_dict(cfg, 0))
    unet = unet.to(dev).eval()
    hin = host_inputs(seed=1000 * rank)
    ns = api.default_schedule()
    ts = torch.linspace(1.0, 1e-3, nfe + 1)
    x_d = hin["x"].to(dev)
    content_d = hin["content"].to(dev).permute(1, 2, 0).contiguous()
    prompt_d = hin["prompt"].to(dev).permute(1, 0, 2).contiguous()
    mask_d = api.sequence_mask(hin["refer_lengths"].to(dev), S)
    gathered = torch.empty((world * B, 100, T), device=dev) if world > 1 else None
    L = _lib.lib()
    h = unet.engine(dev)

    from ns2vc_b200.fused import get_session

    def run_device():
        sess = get_session(unet, content_d, prompt_d, mask_d)
        out = sess.sample_dpmpp_2m(x_d, ns, ts)
        if world > 1:
            gather_latents(out, out=gathered)
            return gathered
        return out

    def run_e2e():
        out = api.sample_latents(unet, hin["x"], hin["content"], hin["prompt"], hin["refer_lengths"], steps=nfe, device=dev)
        if world > 1:
            gather_latents(out, out=gathered)
            return gathered.to("cpu", non_blocking=False) if rank == 0 else out[:1, :1, :1].cpu()
        return out.cpu()

    def timed(fn, K, W, sample_clocks=False):
        for _ in range(W):
            fn()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        cs = ClockSampler(local) if sample_clocks else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            last = fn()
        e1.record()
        torch.cuda.synchronize(dev)
        clocks = cs.stop() if cs else None
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), clocks, last

    ms, clocks, last = timed(run_device, args.steps, args.warmup, sample_clocks=True)
    dumps = {"latents": last.cpu()} if args.dump_outputs and rank == 0 else {}
    # kernel launches per run, counted from the engine's own launch programs (one memset node per
    # forward is not a kernel and is subtracted; +1 sampler-update kernel per step)
    cnt = DenoiserSession(unet, content_d, prompt_d, mask_d)
    cnt.prepare()
    launches_cond = L.ns2vc_unet_launch_count(h)
    cnt.forward(x_d, torch.full((B,), 500.0, device=dev), torch.empty_like(x_d))
    launches_fwd = L.ns2vc_unet_launch_count(h) - 1
    torch.cuda.synchronize(dev)
    del cnt
    units = world * B * nfe * args.steps
    value = units / (ms / 1e3)
    ms_e2e, _, last = timed(run_e2e, args.steps, 1)
    if args.dump_outputs and rank == 0:
        dumps["latents_e2e"] = last
        write_dumps(args.dump_outputs, dumps)
    e2e_val = units / (ms_e2e / 1e3)
    h2d = sum(hin[k].numel() * hin[k].element_size() for k in ("x", "content", "prompt", "refer_lengths"))
    d2h = (world if rank == 0 else 1) * B * 100 * T * 4

    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (3xBF16-split tensor-core contractions, fp32 accumulate)",
           "data": "synthetic", "config": workload_cfg(world), "clocks": clocks,
           "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
           "gpu_launches": ((launches_fwd + 1) * nfe + launches_cond) * args.steps,
           "launches": {"per_unet_forward": launches_fwd, "sampler_update_per_step": 1, "prepare_cond_per_run": launches_cond},
           "ms_per_unet_forward": ms / args.steps / nfe}

    if rank == 0:
        # ---- in-step kernel times: [first CTA entry, last CTA exit] %globaltimer of every launch of ONE forward replayed from a
        # CUDA graph (PDL overlap intact, no event bracketing).  A launch's EXCLUSIVE time = its exit minus max(its entry, the
        # latest exit of the launches before it): the shares add up to the forward, so no kernel can be charged more than the step.
        sess = DenoiserSession(unet, content_d, prompt_d, mask_d)
        sess.prepare()
        tv = torch.full((B,), 500.0, device=dev)
        o = torch.empty_like(x_d)
        for _ in range(2):
            sess.forward(x_d, tv, o)
        torch.cuda.synchronize(dev)
        nl = L.ns2vc_unet_launch_count(h)
        span = torch.empty(nl * 2, dtype=torch.int64, device=dev)
        sv = span.view(nl, 2)
        _lib.check(L.ns2vc_unet_set_span_trace(h, span.data_ptr(), nl))
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            sess.forward(x_d, tv, o)
        _lib.check(L.ns2vc_unet_set_span_trace(h, None, 0))
        g.replay(); torch.cuda.synchronize(dev)
        sv[:, 0] = 0x7fffffffffffffff; sv[:, 1] = 0
        torch.cuda.synchronize(dev)
        g.replay(); torch.cuda.synchronize(dev)
        tr = sv.cpu()
        names = [L.ns2vc_profile_kind_name(L.ns2vc_unet_launch_kind(h, i)).decode() for i in range(nl)]
        rows = [(names[i], int(tr[i, 0]), int(tr[i, 1])) for i in range(nl) if int(tr[i, 1]) > 0]
        excl, dur, cnt = {}, {}, {}
        prev_end = rows[0][1]
        for k, a, e in rows:
            x_us = max(0.0, (e - max(a, prev_end)) / 1e3)
            excl[k] = excl.get(k, 0.0) + x_us; dur[k] = dur.get(k, 0.0) + (e - a) / 1e3; cnt[k] = cnt.get(k, 0) + 1
            prev_end = max(prev_end, e)
        span_us = (max(r[2] for r in rows) - rows[0][1]) / 1e3
        kernels = {k: {"launches_per_forward": cnt[k], "exclusive_us_per_forward": excl[k], "span_sum_us_per_forward": dur[k],
                       "share": excl[k] / span_us} for k in excl}
        del g
        peaks = read_peaks()
        fl_gemm, fl_attn = flops_per_forward(cfg, B, T, S, gemm_only=True)
        fl_gemm += B * 4 * S * cfg.cross_attention_dim * sum(op.cout for op in __import__("ns2vc_b200.arch", fromlist=["build_plan"]).build_plan(cfg) if op.kind == "xformer")  # step-invariant K/V projections (SURVEY 8d counts them)
        gemm_kinds = [k for k in excl if k.startswith("gemm")]                  # every GEMM instantiation (plain / folded-LayerNorm / panel mode) is one kind
        gemm_us, gemm_n = sum(excl[k] for k in gemm_kinds), sum(cnt[k] for k in gemm_kinds)
        dom = "attention" if excl.get("attention", 0.0) > gemm_us else "gemm_tc"
        dom_ms = (excl["attention"] if dom == "attention" else gemm_us) / 1e3
        dom_n = cnt["attention"] if dom == "attention" else gemm_n
        assert dom_ms <= ms / args.steps / nfe * 1.25, "a kernel cannot take longer than the step it is part of"
        if dom == "attention":
            ach = fl_attn / (dom_ms * 1e-3) / 1e12
            alg = f"{fl_attn / 1e9:.1f} GFLOP QK^T+PV per forward"
        else:
            ach = fl_gemm / (dom_ms * 1e-3) / 1e12
            alg = f"{fl_gemm / 1e9:.1f} GFLOP conv+linear per forward (algorithmic, SURVEY 8d; the 3xBF16 split issues 3x this on the tensor pipe); all gemm_tc instantiations"
        traffic = ncu_traffic(dom)
        whole = survey_flops(B, T, S)
        ms_fwd = ms / args.steps / nfe
        t_hbm = SURVEY_BYTES_CFG2 / (peaks["hbm_gbs"] * 1e9) * 1e3
        t_tc = whole / (peaks["tflops"] * 1e12) * 1e3
        out["roofline"] = {"kernel": dom, "bound": "tensor", "achieved": ach, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": ach / peaks["tflops"],
                           "traffic": traffic, "traffic_unit": "DRAM bytes per launch (ncu dram__bytes_read+write, cold-cache capture, profiles/r02_ncu_launches.md)",
                           "algorithmic": alg, "peak_source": peaks["src"], "issued_tflops": 3 * ach if dom == "gemm_tc" else ach,
                           "frac_issued": (3 * ach if dom == "gemm_tc" else ach) / peaks["tflops"],
                           "kernel_ms_per_forward": dom_ms, "launch_avg_us": 1e3 * dom_ms / dom_n,
                           "timing": "exclusive in-step time of the kernel's launches from %globaltimer [entry, exit] spans of one graph-replayed forward (sums to the forward; never above ms_per_unet_forward)",
                           "step": {"ms_per_unet_forward": ms_fwd, "algorithmic_gflop": whole / 1e9, "algorithmic_gb": SURVEY_BYTES_CFG2 / 1e9,
                                    "t_hbm_ms": t_hbm, "t_tc_ms": t_tc, "t_tc_ms_3xbf16_issued": 3 * t_tc,
                                    "binding": "hbm" if t_hbm >= t_tc else "tensor", "frac_vs_binding": max(t_hbm, t_tc) / ms_fwd,
                                    "achieved_tflops": whole / (ms_fwd * 1e-3) / 1e12, "achieved_gbs": SURVEY_BYTES_CFG2 / (ms_fwd * 1e-3) / 1e9,
                                    "note": "SURVEY.md 8(d) constants: 40.20 GFLOP per sample-step (321.6 per cfg2 step), 3.20 GB ideal-fusion bytes; graded against the tighter (larger-time) bound"},
                           "note": "the step is a chain of dependent launches (PDL-linked, one CUDA graph): launches of <= 148 tiles are bound by per-launch latency (TMA round trip, epilogue stores at L2 bandwidth), not by the pipe's FLOP rate"}
        out["kernels"] = kernels
        out["forward_span_us"] = span_us
        # ---- cfg3 (BASELINE.json configs[2]): B=4, T=2048, UniPC bh2 at the reference default of 30 steps and at 50, same process
        try:
            from ns2vc_b200.synth import make_inputs
            c3 = make_inputs(4, 2048, S, seed=3)
            c3s = DenoiserSession(unet, c3["content"].permute(1, 2, 0).contiguous().to(dev), c3["prompt"].permute(1, 0, 2).contiguous().to(dev),
                                  api.sequence_mask(c3["refer_lengths"].to(dev), S))
            x3 = c3["x"].to(dev)
            cfg3 = {}
            for n3 in (30, 50):
                ts3 = torch.linspace(1.0, 1e-3, n3 + 1)
                for _ in range(3):
                    c3s.sample_unipc(x3, ns, ts3)
                torch.cuda.synchronize(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(2):
                    c3s.sample_unipc(x3, ns, ts3)
                e1.record(); torch.cuda.synchronize(dev)
                m3 = e0.elapsed_time(e1) / 2
                cfg3[f"unipc_{n3}"] = {"value": 4 * n3 / (m3 / 1e3), "unit": UNIT, "ms_per_run": m3, "ms_per_unet_forward": m3 / n3}
            out["cfg3"] = {"workload": f"cfg3: B=4, C=100, T=2048, S={S}, UniPC bh2 (order 2), 1 GPU, device-resident inputs", **cfg3}
            del c3s
        except Exception as e:                                   # the extra key must never cost the headline line
            out["cfg3"] = {"error": repr(e)}
        # ---- the condition encoders (Pre_model.infer, the step BEFORE the denoiser: SURVEY.md 8(f) rank 1) at the cfg2 shape,
        # and the whole device pipeline (encoders + 50-NFE sampling) through the public API with host buffers
        try:
            out["pre_model"] = bench_pre_model(unet, dev, hin, nfe, world == 1)
        except Exception as e:
            out["pre_model"] = {"error": repr(e)}
        if world == 1:
            threads = best_thread_count()
            nf = 3
            rate, dt = cpu_oracle_rate(nf, threads)
            out["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                                   "sample": f"{nf} UNet forwards at B={B},T={T},S={S} ({dt:.1f} s) through the oracle port of the reference's CPU PyTorch path, torch threads={threads} (fastest of 8/16/32/64/all on this host; {os.cpu_count()} logical CPUs)"}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
