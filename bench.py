#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric ("ViT frames/sec + LLaMA-13B decode tokens/sec, 8-frame video") on the configuration
it is quoted on.

  N = 1  : BASELINE config 3 -- valley-13b (LLaMA-13B shape, 40 layers) bf16, batch = 4 videos x 8 frames, 256 new tokens.
  N > 1  : BASELINE config 4's per-GPU share on every rank (weak scaling) -- valley-13b, 4 videos x 16 frames per GPU
           (64 frames, 33.7 MB of frame features per rank); the frames of the N*4 videos are DEALT ROUND-ROBIN over the ranks, so
           every rank needs remote frames for the videos it decodes: ViT on the local shard, frame features gathered into every
           rank's buffer by the last ViT GEMM's epilogue (NVLink peer stores; compared bit for bit with NCCL all_gather during
           warm-up), then pool + project + splice + decode of the rank's own 4 videos (LLM replicated).

A *step* is one request batch per rank through the whole hot path: ViT-L/14 encode -> (N>1: gather) -> temporal pool +
mm_projector -> splice -> LLaMA prefill -> greedy decode (one persistent kernel per token, CUDA-graph replay, no host sync).
`value` = generated tokens/s over whole steps, inputs resident in HBM; `e2e` = the same through
ValleyLlamaForCausalLM.generate() (N>1: dist.generate_sharded) from pinned HOST buffers, H2D of pixels + ids and D2H of the token
ids inside the timed region.  The two halves of the metric -- ViT frames/s and steady-state decode tokens/s -- are timed
separately on the device and reported with their roofline fractions (`roofline` = the persistent decode-step kernel the library
launches for this batch -- named in `roofline.kernel` --, HBM; `roofline_vit`).  Every generate call passes eos_token_id=None: exactly
`--new-tokens` decode steps run on every path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model valley-13b|valley2-7b|tiny] [--dump-outputs DIR] ...
  N>1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

--impl reference: the reference algorithm's CPU path (oracle/valley_oracle.py -- plain PyTorch CPU ops, the ATen kernels the
reference's HF modules execute) on this box's host cores; every step is the same BOUNDED SAMPLE of the workload (stated in
`cpu_baseline.sample`), `ms_per_step` is its measured wall time and `value` the whole-request tokens/s it extrapolates to.
"""
from __future__ import annotations

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

from valley_b200 import synthetic as syn  # noqa: E402

GFLOP_PER_FRAME = {-2: 155.29, -1: 162.02}     # BASELINE.md section 3
# committed ncu --set full captures of decode_step_kernel, per (model, batch): dram bytes per launch (profiles/)
NCU_DECODE = {("valley2-7b", 1): "prof_mega_r02_7b_b1_summary.csv", ("valley-13b", 4): "prof_mega_r02_13b_b4_summary.csv",
              ("valley-13b", 1): "prof_mega_r02_13b_b1_summary.csv"}


def prompt_len(n_frames):
    return 1 + 40 + 1 + 256 + 2 + n_frames + 1 + 24


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


def usable_cpus():
    """cpus this process may actually use: affinity mask and cgroup quota, not the machine's core count"""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period) + 0.5)))
    except Exception:
        pass
    return n


def host_memory_budget():
    """bytes this process may allocate: min(MemAvailable, cgroup memory.max - memory.current)"""
    avail = None
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                avail = int(line.split()[1]) * 1024
    except Exception:
        pass
    try:
        mx = open("/sys/fs/cgroup/memory.max").read().strip()
        if mx != "max":
            cur = int(open("/sys/fs/cgroup/memory.current").read())
            room = int(mx) - cur
            avail = room if avail is None else min(avail, room)
    except Exception:
        pass
    return avail if avail is not None else 32 << 30


def cpu_has_bf16_units():
    try:
        flags = open("/proc/cpuinfo").read()
        return ("amx_bf16" in flags) or ("avx512_bf16" in flags)
    except Exception:
        return False


def ncu_traffic(spec_name, B):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of decode_step_kernel from the committed ncu --set full capture of
    THIS (model, batch) -- None when no capture of that configuration is committed."""
    name = NCU_DECODE.get((spec_name, B))
    if not name:
        return None, None
    try:
        import csv
        rows = list(csv.reader(open(os.path.join(ROOT, "profiles", name))))
        hdr, units, row = rows[0], rows[1], rows[2]
        tot = 0.0
        for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            i = hdr.index(k)
            tot += float(row[i]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}.get(units[i], 1.0)
        return tot, "profiles/" + name
    except Exception:
        return None, None


def decode_bytes_per_step(spec, B, S):
    """Algorithmic HBM bytes of one decode step (SURVEY 8d): every weight once (bf16) + KV read + KV write."""
    H, I, V, L = spec.hidden_size, spec.intermediate_size, spec.vocab_size, spec.num_hidden_layers
    w = 2 * (L * (4 * H * H + 3 * H * I) + V * H)
    kv = B * S * 2 * L * H * 2 + B * 2 * L * H * 2
    return w + kv


def gather_rows(x, world):
    """every rank's rows of ``x`` (equal shapes), in rank order: the whole batch on every rank"""
    if world == 1:
        return x
    import torch.distributed as dist
    parts = [torch.empty_like(x) for _ in range(world)]
    dist.all_gather(parts, x.contiguous())
    return torch.cat(parts)


DUMP_CAP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, rank=0):
    """rank 0 writes each tensor as out_dir/<name>.npy in float64; an array past DUMP_CAP_BYTES is cut to a fixed, seeded
    sample of its rows so that all files together stay under the cap"""
    if rank != 0:
        return
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_CAP_BYTES // max(len(arrays), 1)
    for name, x in arrays.items():
        x = x.detach().cpu().double().numpy()
        if x.nbytes > budget:
            keep = max(1, budget // max(x[0].nbytes, 1))
            x = x[np.sort(np.random.default_rng(0).choice(len(x), keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), x)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm's CPU path (oracle port), one bounded sample per step, all usable host threads
# ------------------------------------------------------------------------------------------------------
class CpuReferenceArm:
    """The reference's algorithm on the host cores: oracle/valley_oracle.py == the ATen CPU ops its HF modules run.

    One *sample step* (the same every step, wall-clocked as a whole):
        ViT-L/14 at full depth on ONE video's frames                                         -> t_vit
        LLaMA prefill of ONE prompt row (S tokens) through ALL layers + lm_head (last row)   -> t_prefill
        n_dec decode steps at the workload's batch B through ALL layers + lm_head + argmax   -> t_dec (per step)
    The B videos / rows of a request are independent on a CPU (no cross-row reuse beyond what the batched decode step already
    has), so the whole request is  B t_vit + B t_prefill + (n_new - 1) t_dec  and tokens/s = B n_new / that.
    Thread count = the cpus this process may use (affinity & cgroup quota), fixed.  Precision = bf16 when the CPU has bf16
    matrix units (AMX / AVX512-BF16: what a user of the reference would run), else fp32; fixed per box, not re-probed.
    Weights: ONE layer of random-init tensors, cloned per layer -- distinct memory for every layer (a decode step streams the
    full model from DRAM) without paying 13 G random draws; values do not influence the timing.  If the host cannot hold the full
    depth, the deepest stack that fits is timed and the layer time is scaled (said in `sample`)."""

    def __init__(self, spec, B, T, n_new, n_dec=2):
        import dataclasses
        from oracle import valley_oracle as O
        self.O, self.spec, self.B, self.T, self.n_new, self.n_dec = O, spec, B, T, n_new, n_dec
        self.threads = usable_cpus()
        torch.set_num_threads(self.threads)
        self.dtype = torch.bfloat16 if cpu_has_bf16_units() else torch.float32
        self.S = prompt_len(T)
        L = spec.num_hidden_layers
        H, I, V = spec.hidden_size, spec.intermediate_size, spec.vocab_size
        esz = 2 if self.dtype == torch.bfloat16 else 4
        per_layer = (4 * H * H + 3 * H * I) * esz
        fixed = 2 * V * H * esz + 700e6 * esz / 2 + (4 << 30)            # embed + lm_head + ViT + working set
        room = host_memory_budget() * 0.8 - fixed
        self.layers = int(max(1, min(L, room // per_layer)))
        t0 = time.time()
        one = dataclasses.replace(spec, num_hidden_layers=1)
        self.vit_w = {k: v.to(self.dtype) for k, v in syn.iter_state_dict(spec, 0, llm=False)}
        base = {k: v.to(self.dtype) for k, v in syn.iter_state_dict(one, 0, vision=False)}
        self.llm_w = {k: v for k, v in base.items() if not k.startswith("model.layers.")}
        for i in range(self.layers):
            for k, v in base.items():
                if k.startswith("model.layers.0."):
                    self.llm_w[k.replace("model.layers.0.", f"model.layers.{i}.")] = v if i == 0 else v.clone()
        self.px = syn.make_pixels(1, T, 0)[0].to(self.dtype)
        self.emb_row = (torch.randn(1, self.S, H) * 0.5).to(self.dtype)
        self.emb_dec = (torch.randn(B, 1, H) * 0.5).to(self.dtype)
        self.setup_s = time.time() - t0
        self.kw = dict(n_layers=self.layers, heads=spec.num_attention_heads, eps=spec.rms_norm_eps)

    def step(self):
        """one bounded sample; returns its wall time and the three component times"""
        O, spec = self.O, self.spec
        lin = torch.nn.functional.linear
        t_all = time.perf_counter()
        with torch.no_grad():
            t = time.perf_counter()
            O.vit_hidden_state(self.vit_w, self.px, spec.mm_vision_select_layer, num_layers=spec.vit_layers)
            t_vit = time.perf_counter() - t
            cache = O.KVCache(self.layers)
            t = time.perf_counter()
            h = O.llama_model(self.llm_w, self.emb_row, cache, **self.kw)
            lin(h[:, -1:], self.llm_w["lm_head.weight"]).argmax(-1)
            t_pre = time.perf_counter() - t
            # decode at batch B: the cache holds the prompt of every row
            for l in range(self.layers):
                cache.k[l] = cache.k[l].expand(self.B, -1, -1, -1).contiguous()
                cache.v[l] = cache.v[l].expand(self.B, -1, -1, -1).contiguous()
            t = time.perf_counter()
            for _ in range(self.n_dec):
                hh = O.llama_model(self.llm_w, self.emb_dec, cache, **self.kw)
                lin(hh, self.llm_w["lm_head.weight"]).argmax(-1)
            t_dec = (time.perf_counter() - t) / self.n_dec
        return dict(wall=time.perf_counter() - t_all, t_vit=t_vit, t_prefill=t_pre, t_dec=t_dec)

    def extrapolate(self, r):
        """whole-request figures from one sample (layer time scaled only if the full depth did not fit in host memory)"""
        L, k = self.spec.num_hidden_layers, self.spec.num_hidden_layers / self.layers
        t_pre = r["t_prefill"] * k if self.layers < L else r["t_prefill"]
        t_dec = r["t_dec"] * k if self.layers < L else r["t_dec"]
        total = self.B * r["t_vit"] + self.B * t_pre + (self.n_new - 1) * t_dec
        return dict(tokens_per_s=self.B * self.n_new / total, vit_frames_per_s=self.T / r["t_vit"], decode_tokens_per_s=self.B / t_dec,
                    prefill_s_per_row=t_pre, request_s=total)

    def describe(self):
        L = self.spec.num_hidden_layers
        nm = {torch.bfloat16: "bf16", torch.float32: "fp32"}[self.dtype]
        depth = f"all {L} layers" if self.layers == L else f"{self.layers} of {L} layers (host memory bound; layer time scaled x{L / self.layers:.2f})"
        return (f"oracle port on {self.threads} host threads (usable cpus; machine reports {os.cpu_count()}), {nm}; per step: ViT-L/14 "
                f"({self.spec.vit_layers + 1 + self.spec.mm_vision_select_layer} layers) on {self.T} frames of one video + prefill of one {self.S}-token row "
                f"through {depth} + lm_head + {self.n_dec} decode steps at batch {self.B} through {depth} + lm_head; "
                f"request = {self.B} x ViT + {self.B} x prefill row + {self.n_new - 1} x decode step")


def gpu_eager_reference(spec, B, n_frames, n_new, decode_tokens=16):
    """SURVEY 8d "reference GPU path": the same oracle (the ATen ops the reference's HF modules run, eager, bf16) on the B200 itself.
    Not a target and not the product -- it says how much of the speed-up is the GPU and how much is this repo."""
    from oracle import valley_oracle as O
    dev, dt = "cuda", torch.bfloat16
    w = dict(syn.iter_state_dict(spec, 0, device=dev, dtype=dt))
    S = prompt_len(n_frames)
    px = syn.make_pixels(1, B * n_frames, 0)[0].to(dev, dt)
    kw = dict(n_layers=spec.num_hidden_layers, heads=spec.num_attention_heads, eps=spec.rms_norm_eps)

    def ev():
        return torch.cuda.Event(enable_timing=True)
    with torch.no_grad():
        for _ in range(2):
            O.vit_hidden_state(w, px, spec.mm_vision_select_layer, num_layers=spec.vit_layers)
        e0, e1 = ev(), ev()
        e0.record()
        for _ in range(3):
            O.vit_hidden_state(w, px, spec.mm_vision_select_layer, num_layers=spec.vit_layers)
        e1.record()
        torch.cuda.synchronize()
        ms_vit = e0.elapsed_time(e1) / 3
        emb = torch.randn(B, S, spec.hidden_size, device=dev).to(dt)
        cache = O.KVCache(spec.num_hidden_layers)
        e0, e1 = ev(), ev()
        e0.record()
        h = O.llama_model(w, emb, cache, **kw)
        tok = torch.nn.functional.linear(h[:, -1:], w["lm_head.weight"]).argmax(-1)
        e1.record()
        torch.cuda.synchronize()
        ms_prefill = e0.elapsed_time(e1)

        def step(tok):
            x = torch.nn.functional.embedding(tok, w["model.embed_tokens.weight"])
            hh = O.llama_model(w, x, cache, **kw)
            return torch.nn.functional.linear(hh, w["lm_head.weight"]).argmax(-1)
        for _ in range(3):
            tok = step(tok)
        e0, e1 = ev(), ev()
        e0.record()
        for _ in range(decode_tokens):
            tok = step(tok)
            tok[0].item()                                      # the reference syncs device->host every token (model_worker.py:390)
        e1.record()
        torch.cuda.synchronize()
        ms_dec = e0.elapsed_time(e1) / decode_tokens
    del w
    torch.cuda.empty_cache()
    total = ms_vit + ms_prefill + (n_new - 1) * ms_dec
    return {"what": "oracle (eager torch ops, bf16) on the same B200", "tokens_per_s": B * n_new / (total / 1e3), "vit_frames_per_s": B * n_frames / (ms_vit / 1e3),
            "prefill_ms": ms_prefill, "decode_ms_per_step": ms_dec, "decode_tokens_per_s": B * 1e3 / ms_dec}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="valley-13b", choices=list(syn.SPECS))
    ap.add_argument("--batch", type=int, default=4, help="videos per GPU (BASELINE config 3 / 4: 4)")
    ap.add_argument("--new-tokens", type=int, default=256)
    ap.add_argument("--frames", type=int, default=None, help="frames per video; default 8 at N = 1 (config 3), 16 at N > 1 (config 4)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-7b", action="store_true", help="skip the extra valley2-7b B=1 figures (BASELINE config 2)")
    ap.add_argument("--vit-sweep", action="store_true", help="also time ViT encode over F (BASELINE config 5); N > 1: strong scaling, F fixed")
    ap.add_argument("--gpu-eager-baseline", action="store_true", help="also time the oracle as eager torch-CUDA ops on the GPU (SURVEY 8d)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (the generated token ids of every "
                         "sequence) to DIR/<name>.npy as float64, for comparing two builds output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    spec = syn.SPECS[a.model]
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    T = a.frames if a.frames is not None else (8 if a.gpus <= 1 else 16)
    N_NEW, B = a.new_tokens, a.batch
    S = prompt_len(T)
    metric = f"generated tokens/s ({T}-frame video requests: ViT-L/14 encode + pool/project + LLaMA prefill + {N_NEW} greedy tokens per sequence)"
    cfg_common = {
        "workload": f"{a.model} bf16: {B} videos x {T} frames 224x224 per GPU ({B * T} frames/GPU), prompt S={S}, greedy {N_NEW} new tokens per sequence"
                    + (" [BASELINE config 3]" if (a.gpus <= 1 and a.model == "valley-13b" and B == 4 and T == 8) else "")
                    + (" [BASELINE config 4 per-GPU share, weak scaling]" if (a.gpus > 1 and a.model == "valley-13b" and B == 4 and T == 16) else ""),
        "batch_per_gpu": B, "frames": T, "new_tokens": N_NEW,
        "parallelism": f"dp{a.gpus}" + ("" if a.gpus <= 1 else " (frames dealt round-robin over ranks -> every rank needs remote frames; frame features gathered by the "
                                        "last ViT GEMM epilogue via NVLink peer stores; LLM replicated, each rank decodes its own videos)"),
        "l2": f"inputs larger than L2 ({2 * (spec.num_hidden_layers * (4 * spec.hidden_size ** 2 + 3 * spec.hidden_size * spec.intermediate_size) + spec.vocab_size * spec.hidden_size) / 1e9:.1f} GB "
              "of weights stream per decode step; ViT weights 606 MB)",
        "stopping": f"eos stopping disabled (eos_token_id=None): every sequence runs exactly {N_NEW} decode steps on every path"}

    if a.impl == "reference":
        if rank != 0:
            return
        arm = CpuReferenceArm(spec, B, T, N_NEW)
        for _ in range(a.warmup):
            arm.step()
        t0 = time.perf_counter()
        rs = [arm.step() for _ in range(a.steps)]
        wall = time.perf_counter() - t0
        ex = [arm.extrapolate(r) for r in rs]
        v = statistics.median(e["tokens_per_s"] for e in ex)
        print(json.dumps({
            "impl": "reference", "metric": metric, "value": v, "unit": "tokens/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1e3 * wall / max(a.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {torch.bfloat16: "bf16", torch.float32: "f32"}[arm.dtype], "data": "synthetic", "config": cfg_common,
            "value_is": "median over the timed steps of the whole-request tokens/s each step's bounded sample extrapolates to; ms_per_step is the "
                        "measured wall time of one sample step",
            "vit_frames_per_s": statistics.median(e["vit_frames_per_s"] for e in ex),
            "decode_tokens_per_s": statistics.median(e["decode_tokens_per_s"] for e in ex),
            "prefill_s_per_row": statistics.median(e["prefill_s_per_row"] for e in ex),
            "per_step": [{k: round(x, 4) for k, x in r.items()} for r in rs], "setup_s": arm.setup_s,
            "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": arm.threads, "kind": "port", "sample": arm.describe()},
            "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # ------------------------------------------------------------------ ours
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    import torch.distributed as dist
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line (NCCL prints its version banner there)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    import ctypes as C
    from valley_b200 import dist as vdist
    from valley_b200._lib import VlySampling, check
    from valley_b200.model import ValleyConfig, ValleyLlamaForCausalLM

    def load(spec_):
        t0 = time.time()
        m = ValleyLlamaForCausalLM(ValleyConfig.from_spec(spec_), local)
        m.load_state_dict(syn.iter_state_dict(spec_, 0, device=f"cuda:{local}"))
        for k, v in syn.sentinel_ids(spec_).items():
            setattr(m.get_model().vision_tower.config, k, v)
        torch.cuda.synchronize()
        return m, time.time() - t0
    model, t_load = load(spec)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, K, W, mdl=None):
        mdl = mdl or model
        for _ in range(W):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = mdl.launches()
        e0.record()
        for _ in range(K):
            r = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms / K, mdl.launches() - l0, r

    n_videos = world * B                           # weak scaling: B videos per GPU
    F_total = n_videos * T
    ids_all = syn.make_prompt_ids(spec, n_videos, T, 0)
    px_all = syn.make_pixels(n_videos, T, 0, dtype=torch.float16).reshape(F_total, 3, 224, 224)     # callers send fp16 pixels (valley_model.py:430)
    vlo, vhi = vdist.shard_bounds(n_videos, world, rank)
    mine = list(vdist.dealt_frames(F_total, world, rank)) if world > 1 else list(range(F_total))
    px_local_host = px_all[mine].contiguous().pin_memory()
    ids_host = ids_all[vlo:vhi].contiguous().pin_memory()
    px_dev, ids_dev = px_local_host.cuda(non_blocking=True), ids_host.cuda(non_blocking=True)
    fused = None
    if world > 1:      # one gather buffer per context: sized for the largest encode of this run, used for F_total frames by default
        fused = vdist.FusedFrameGather(model, max(F_total, 4096 if a.vit_sweep else 0))
        fused.n_frames_total = F_total

    def step_device():
        if world > 1:
            return vdist.generate_sharded(model, ids_dev, px_dev, n_videos, T, N_NEW, fused=fused, interleaved=True)
        return model.generate(input_ids=ids_dev, images=px_dev.view(B, T, 3, 224, 224), max_new_tokens=N_NEW, eos_token_id=None)[:, S:]

    def step_e2e():
        px = px_local_host.cuda(non_blocking=True)
        ids = ids_host.cuda(non_blocking=True)
        if world > 1:
            out = vdist.generate_sharded(model, ids, px, n_videos, T, N_NEW, fused=fused, interleaved=True)
        else:
            out = model.generate(input_ids=ids, images=px.view(B, T, 3, 224, 224), max_new_tokens=N_NEW, eos_token_id=None)[:, S:]
        return out.cpu()

    if os.environ.get("VLY_BENCH_PROFILE"):
        # ncu launch list of exactly the timed step:  ncu --profile-from-start off --metrics gpu__time_duration.sum ... bench.py
        for _ in range(max(a.warmup, 3)):
            step_device()
        barrier()
        torch.cuda.profiler.start()
        step_device()
        barrier()
        torch.cuda.profiler.stop()
        print(json.dumps({"profiled": "one timed step", "launches": int(model.launches())}))
        return

    # ---- multi-GPU correctness of the path that is about to be timed (warm-up; VERDICT r1 #1) ----
    multi = {}
    if world > 1:
        got = fused.encode(px_dev, True)
        torch.cuda.synchronize()
        ref = vdist.encode_frames_sharded(model.encode_frames, px_dev, F_total, interleaved=True)       # local ViT + NCCL all_gather
        same = torch.tensor([1 if torch.equal(got, ref) else 0], device="cuda")
        fused.release()
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        # this rank's tokens from the sharded path vs a single-GPU run of the same videos (all of their frames encoded locally)
        toks_sharded = step_device()
        own_px = px_all.view(n_videos, T, 3, 224, 224)[vlo:vhi].cuda()
        toks_single = model.generate(input_ids=ids_dev, images=own_px, max_new_tokens=N_NEW, eos_token_id=None)[:, S:]
        tm = torch.tensor([1 if torch.equal(toks_sharded, toks_single) else 0], device="cuda")
        dist.all_reduce(tm, op=dist.ReduceOp.MIN)
        fused.check()
        multi = {"gather_bit_identical": bool(same.item()), "tokens_match_n1": bool(tm.item()), "gather_timeout_flag": False}
        del ref, own_px

    clk = ClockSampler(local)
    if rank == 0:
        clk.start()
    ms_step, launches, toks = timed(step_device, a.steps, max(a.warmup, 3))
    clocks = clk.stop() if rank == 0 else None
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"tokens": gather_rows(toks, world)}, rank)
    ms_e2e, _, toks_e2e = timed(step_e2e, a.steps, 1)

    # ---- the two halves of the metric, timed separately on the device ----
    def vit_only(F, mdl=None):
        px = syn.make_pixels(1, F, 1, dtype=torch.float16)[0].cuda()
        return timed(lambda: (mdl or model).encode_frames(px), max(a.steps, 5), 3, mdl)[0]
    F_req = B * T
    ms_vit_req = vit_only(F_req)
    ms_vit8 = vit_only(8) if F_req != 8 else ms_vit_req
    sweep = {}
    if a.vit_sweep and world == 1:
        for F in (1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096):
            sweep[str(F)] = F / (vit_only(F) / 1e3)

    if world > 1:
        # cost of the collective: fused encode+gather vs the same local encode without it, and the plain NCCL all_gather alone
        ms_fused = timed(lambda: (fused.encode(px_dev, True), fused.release()), 5, 2)[0]
        ms_local = timed(lambda: model.encode_frames(px_dev), 5, 2)[0]
        feats_local = model.encode_frames(px_dev)
        ms_nccl = timed(lambda: vdist.gather_frame_features(feats_local, F_total, interleaved=True), 5, 2)[0]
        sent = (world - 1) * feats_local.numel() * 2
        multi.update({"vit_fused_gather_ms": ms_fused, "vit_local_only_ms": ms_local, "gather_ms": max(ms_fused - ms_local, 0.0),
                      "nccl_allgather_ms": ms_nccl, "gather_bytes_sent_per_rank": int(sent), "gather_bytes_received_per_rank": int(sent),
                      # (None: the peer stores ride inside the last GEMM's epilogue -- no measurable cost to divide by)
                      "gather_gbs_per_rank_if_not_hidden": (sent / (ms_fused - ms_local) / 1e6) if ms_fused - ms_local > 0.01 else None,
                      "nccl_gbs_per_rank": sent / ms_nccl / 1e6})
        fused.check()
        del feats_local
        if a.vit_sweep:      # BASELINE config 5 across GPUs: STRONG scaling -- F fixed, frames dealt round-robin, fused gather included
            strong = {}
            for F in (1024, 4096):
                fused.n_frames_total = F
                n_loc = len(vdist.dealt_frames(F, world, rank))
                pxs = syn.make_pixels(1, n_loc, 1 + rank, dtype=torch.float16)[0].cuda()
                ms = timed(lambda: (fused.encode(pxs, True), fused.release()), 5, 2)[0]
                strong[str(F)] = F / (ms / 1e3)
                del pxs
            fused.n_frames_total = F_total
            multi["vit_strong_scaling_frames_per_s"] = strong
            fused.check()

    def llm_only(mdl, spec_, B_, T_, n_new):
        """steady-state decode ms/step, prefill ms, sampled-decode ms/step of one model"""
        ids = syn.make_prompt_ids(spec_, B_, T_, 0).cuda()
        S_ = ids.shape[1]
        _, _, _, emb, _ = mdl.prepare_inputs_labels_for_multimodal(ids, None, None, None, None)
        cache = mdl.new_cache(B_)
        _, nxt = mdl._prefill(cache, emb, 0)
        out = torch.empty(B_, n_new, dtype=torch.int64, device="cuda")
        st = lambda: torch.cuda.current_stream().cuda_stream

        def run(n):
            check(mdl._lib.vly_generate_greedy(mdl._ctx, cache._h, nxt.data_ptr(), n, out.data_ptr(), st()))
        run(8)                                    # warm-up incl. graph capture
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(n_new - 8)
        e1.record()
        barrier()
        ms_dec = e0.elapsed_time(e1) / (n_new - 8)
        s_mid = S_ + 8 + (n_new - 8) / 2

        def f():
            cache.reset()
            mdl._prefill(cache, emb, 0)
        ms_pre = timed(f, 3, 2, mdl)[0]
        # the same steady-state decode with temperature sampling + eos bookkeeping selected inside the step (f-1)
        cache.reset()
        _, nxt2 = mdl._prefill(cache, emb, 0)
        sp = VlySampling(0.8, 1234, spec_.vocab_size + 5, 0)          # an eos id that can never be drawn: bookkeeping on, no early stop

        def run_s(n):
            check(mdl._lib.vly_generate(mdl._ctx, cache._h, nxt2.data_ptr(), n, out.data_ptr(), C.byref(sp), None, st()))
        run_s(8)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run_s(n_new - 8)
        e1.record()
        barrier()
        return ms_dec, s_mid, ms_pre, e0.elapsed_time(e1) / (n_new - 8), cache.decode_kernel()
    ms_dec, s_mid, ms_prefill, ms_dec_sampled, dec_kernel = llm_only(model, spec, B, T, N_NEW)

    def preprocess_only():
        """f-2: 8 decoded 720p uint8 frames -> [8,3,224,224] fp16 (device-resident input; and from pinned host memory)"""
        from valley_b200 import video
        g = torch.Generator().manual_seed(5)
        host = torch.randint(0, 256, (8, 720, 1280, 3), dtype=torch.uint8, generator=g).pin_memory()
        dev = host.cuda()
        return timed(lambda: video.preprocess_frames(model, dev), 20, 3)[0], timed(lambda: video.preprocess_frames(model, host), 20, 3)[0], host
    ms_pre_dev, ms_pre_host, pre_host = preprocess_only()

    # extra: BASELINE config 2 (valley2-7b, one 8-frame video, 128 tokens) on the same GPU, N = 1 only
    cfg2 = None
    if world == 1 and not a.no_7b and a.model != "valley2-7b":
        free = torch.cuda.mem_get_info()[0]
        if free > 40e9:
            s7 = syn.VALLEY2_7B
            m7, _ = load(s7)
            ids7 = syn.make_prompt_ids(s7, 1, 8, 0).cuda()
            px7 = syn.make_pixels(1, 8, 0, dtype=torch.float16).cuda()
            S7 = ids7.shape[1]
            ms7, l7, _ = timed(lambda: m7.generate(input_ids=ids7, images=px7, max_new_tokens=128, eos_token_id=None)[:, S7:], 3, 2, m7)
            d7, smid7, p7, _, k7 = llm_only(m7, s7, 1, 8, 128)
            b7 = decode_bytes_per_step(s7, 1, smid7)
            tr7, src7 = ncu_traffic("valley2-7b", 1)
            cfg2 = {"workload": "valley2-7b bf16: 1 video x 8 frames, prompt S=333, greedy 128 new tokens [BASELINE config 2]",
                    "tokens_per_s": 128 / (ms7 / 1e3), "ms_per_request": ms7, "gpu_launches_per_request": int(l7 / 3),
                    "decode_ms_per_token": d7, "decode_tokens_per_s": 1e3 / d7, "prefill_ms": p7,
                    "roofline": {"kernel": k7, "bound": "hbm", "achieved": b7 / (d7 / 1e3) / 1e9, "peak": peaks()["hbm"], "unit": "GB/s",
                                 "frac": b7 / (d7 / 1e3) / 1e9 / peaks()["hbm"], "algorithmic_bytes_per_launch": b7, "traffic": tr7, "traffic_source": src7}}
            del m7
            torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    value = world * B * N_NEW / (ms_step / 1e3)
    e2e = world * B * N_NEW / (ms_e2e / 1e3)
    dec_bytes = decode_bytes_per_step(spec, B, s_mid)
    dec_gbs = dec_bytes / (ms_dec / 1e3) / 1e9
    fps_req = F_req / (ms_vit_req / 1e3)
    fps8 = 8 / (ms_vit8 / 1e3)
    gf = GFLOP_PER_FRAME.get(spec.mm_vision_select_layer, 155.29) if spec.vit_layers == 24 else None
    traffic, traffic_src = ncu_traffic(a.model, B)
    line = {
        "metric": metric, "value": value, "unit": "tokens/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic (random-init weights of the named architecture, N(0,1) pixels, seeded prompt ids)",
        "config": cfg_common,
        "e2e": {"value": e2e, "unit": "tokens/s", "h2d_bytes_per_step": int(px_local_host.numel() * 2 + ids_host.numel() * 8),
                "d2h_bytes_per_step": int(B * N_NEW * 8), "ms_per_step": ms_e2e,
                "api": ("valley_b200.dist.generate_sharded(model, ids, pixels, ...)" if world > 1 else "ValleyLlamaForCausalLM.generate(input_ids, images)") + " from pinned host tensors"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "decode_tokens_per_s": world * B / (ms_dec / 1e3), "decode_ms_per_step": ms_dec, "decode_batch": B,
        "vit_frames_per_s": world * fps_req, "vit_frames_per_encode": F_req, "vit_ms_per_encode": ms_vit_req,
        "vit_frames_per_s_at_8_frames": world * fps8, "prefill_ms": ms_prefill, "vit_sweep_frames_per_s": sweep,
        "roofline": {"kernel": f"{dec_kernel} (one persistent cooperative launch = one decode step of all {B} sequences: every weight streamed once through a TMA ring"
                               + ("; tcgen05 consumer" if "umma" in dec_kernel else "") + ")",
                     "bound": "hbm", "achieved": dec_gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": dec_gbs / pk["hbm"], "peak_source": pk["src"],
                     "algorithmic_bytes_per_launch": dec_bytes, "traffic": traffic, "traffic_source": traffic_src,
                     "note": "peak = measured read+write copy bandwidth; a read-only stream on this part reaches 7.2-7.5 TB/s (tools/membw.cu)"},
        "roofline_vit": None if gf is None else {
            "kernel": f"ViT-L/14 encode (gemm_tc_kernel + vit_attention_pp_kernel), F={F_req} (the request's frames in one encode)", "bound": "tensor",
            "achieved": fps_req * gf / 1e3, "peak": pk["tf_burst"], "unit": "TFLOP/s", "frac": fps_req * gf / 1e3 / pk["tf_burst"],
            "frac_at_8_frames": fps8 * gf / 1e3 / pk["tf_burst"], "gflop_per_frame": gf, "peak_source": pk["src"],
            "sweep_frac_of_sustained": {k: v * gf / 1e3 / pk["tf_sust"] for k, v in sweep.items()}},
        "decode_sampled_ms_per_step": ms_dec_sampled,
        "preprocess": {"workload": "8 frames 720x1280x3 uint8 -> Resize(256, PIL bilinear) -> CenterCrop(224) -> CLIP normalise -> [8,3,224,224] fp16",
                       "frames_per_s": world * 8 / (ms_pre_dev / 1e3), "ms_8_frames": ms_pre_dev,
                       "e2e_frames_per_s": world * 8 / (ms_pre_host / 1e3), "e2e_ms_8_frames": ms_pre_host, "h2d_bytes": int(pre_host.numel())},
        "weights_load_s": t_load,
        "tokens_match_e2e": bool(torch.equal(toks.cpu(), toks_e2e)),
    }
    line.update(multi)
    if cfg2 is not None:
        line["config2_valley2_7b_b1"] = cfg2
    if not a.no_cpu_baseline:
        arm = CpuReferenceArm(spec, B, T, N_NEW)
        arm.step()                                                            # warm-up (first-touch, thread pool)
        rs = [arm.step() for _ in range(3)]
        ex = [arm.extrapolate(r) for r in rs]
        med = lambda k: statistics.median(e[k] for e in ex)
        line["cpu_baseline"] = {"value": med("tokens_per_s"), "unit": "tokens/s", "cores": arm.threads, "kind": "port", "sample": arm.describe(),
                                "repetitions": 3, "statistic": "median", "sample_wall_s": [round(r["wall"], 3) for r in rs],
                                "vit_frames_per_s": med("vit_frames_per_s"), "decode_tokens_per_s": med("decode_tokens_per_s"),
                                "prefill_s_per_row": med("prefill_s_per_row")}
        from oracle import preprocess_oracle as PO          # the reference's PIL pipeline, executed by Pillow (1 core, as load_video runs it)
        t0 = time.perf_counter()
        for _ in range(3):
            PO.pil_pipeline(pre_host.numpy())
        line["cpu_baseline"]["preprocess_frames_per_s"] = 3 * 8 / (time.perf_counter() - t0)
    if a.gpu_eager_baseline:
        line["gpu_eager_baseline"] = gpu_eager_reference(spec, B, T, N_NEW)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
