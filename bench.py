#!/usr/bin/env python
"""bench.py — the hot path of BASELINE.json: Task reconciles through `provider: local`.

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic Task CRs: BASELINE config 2 (the
largest single-GPU configuration, the one nearest north_star's ">= 1000 concurrent Task CRs"):
512 concurrent Tasks, context windows log-uniform on [128, 4096] tokens (seeded, mean ~1150),
continuous batching, greedy, max_tokens 64, Llama-3-8B shapes with seeded synthetic bf16 weights (no
checkpoints or network in this image).  Config 1 (64 Tasks x 512 tokens) is run on the same engine
after the timed region and reported under the extra key "config1".  Every Task goes  Task CR JSON -> sendLLMRequest (C++ mirror of the reference's
Task step) -> LLMClient.SendRequest -> C ABI (host JSON in, host JSON out) -> continuous-batching
CUDA engine -> assistant message -> processLLMResponse -> status writes.

Reported on ONE JSON line (rank 0):
  metric  task_reconciles_per_s          (BASELINE.json: "Task reconciles/sec and decode tokens/sec")
  value   reconciles / device-timed seconds (CUDA events around every prefill/decode step; inputs
          already resident: weights + KV in HBM)
  e2e     the same reconciles / wall seconds measured around the host call, host buffers,
          H2D (step descriptors, page tables, token ids) and D2H (sampled tokens) inside
  decode_tokens_per_s, p50/p99_decode_step_ms, roofline (algorithmic HBM bytes per decode step /
  device time per decode step vs MEASURED_PEAKS.json hbm_gbs), roofline_prefill (algorithmic FLOPs of
  the prefill steps incl. causal attention / their device time vs bf16_tflops_sustained), cpu_baseline (the reference's CPU reconcile
  loop restated in C++ against a loopback stub completion server, same box, core count stated).

N > 1: one engine replica per GPU (request-level data parallelism, no collective on the data
path — DESIGN.md §6); weak scaling: every rank runs its own 64 Tasks; time = max over ranks.

--impl reference: the reference's own path for this metric is a CPU reconcile loop doing HTTP to
a provider; it cannot be built here (Go, no toolchain), so the arm runs the C++ restatement
(agentcontrolplane_b200/csrc/host, provider "openai" over loopback to the stub server returning
the reference's fixture body) on all host cores, on rank 0 only.  That restatement lives in its own
library, libacp_host.so (pure C++, not linked against the product): the reference arm never maps
libacp_infer.so.

--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step handed back to the Tasks'
owner, DIR/task_output_bytes.npy: float32 [tasks, width], row i = the UTF-8 bytes of Task i's status.output,
padded with -1.  width = 5 * max_tokens (a synthetic token decodes to at most 5 bytes), so the shape does not
depend on what was generated.  Step i always runs seed i + 1: the same arguments give the same inputs, and
two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only: the benchmark writes nothing into it

WORKLOADS = {
    # BASELINE.json configs[2]: the largest single-GPU configuration (default since round 2)
    2: {"name": "llama-3-8b provider:local, 512 concurrent Task CRs, context windows log-uniform 128..4096 tokens (mean ~1150), "
                "continuous batching, greedy, max_tokens 64",
        "model": "llama-3-8b", "tasks": 512, "prompt_tokens": 0, "prompt_min": 128, "prompt_max": 4096, "max_tokens": 64,
        "tp": 1, "tools": 0, "tool_loop": False},
    # BASELINE.json configs[1]: 64 Tasks x 512 tokens (round 1's driver line; now the "config1" extra key)
    1: {"name": "llama-3-8b provider:local, 64 concurrent Task CRs, 512-token context, greedy, max_tokens 64",
        "model": "llama-3-8b", "tasks": 64, "prompt_tokens": 512, "max_tokens": 64, "tp": 1, "tools": 0, "tool_loop": False},
    # BASELINE.json configs[3]: 70B tensor-parallel over 8 GPUs of ONE process, tool-call loop
    # (2 LLM steps per Task: scripted tool call -> ToolCall CR "executes" -> fold-back -> final answer)
    3: {"name": "llama-3-70b TP=8 provider:local, 256 concurrent Task CRs with tool-call loop, 512-token context, greedy, max_tokens 64",
        "model": "llama-3-70b", "tasks": 256, "prompt_tokens": 512, "max_tokens": 64, "tp": 8, "tools": 2, "tool_loop": True},
    # BASELINE.json configs[4]: Mixtral-8x7B, experts spread over the 8 GPUs of ONE process (expert parallel on the
    # tensor-parallel ranks), open-loop Poisson arrivals at 1024 Tasks/s, every root Task delegates down a depth-2
    # sub-agent chain (5 LLM steps + 2 ToolCall CRs + 2 child Task CRs per root Task)
    4: {"name": "mixtral-8x7b EP=8 provider:local, Poisson arrivals 1024 Tasks/s for 1 s (1024 root Tasks), depth-2 sub-agent "
                "delegation chains, 512-token root windows, greedy, max_tokens 64",
        "model": "mixtral-8x7b", "tasks": 1024, "prompt_tokens": 512, "max_tokens": 64, "tp": 8, "tools": 0, "tool_loop": False,
        "arrival_rate": 1024.0, "delegation_depth": 2},
}
WORKLOAD = WORKLOADS[2]
# DRAM bytes of ONE decode step from the committed `ncu --set full` captures (dram__bytes_read + write)
NCU_TRAFFIC = {1: 20.00e9, 2: 107.4e9}
NCU_TRAFFIC_SOURCE = {1: "profiles/r1_v3_ncu_full_decode_kernels.md: 32 x (QKV 51.2 + attention 146.0 + O 34.1 "
                         "+ gate/up 238.4 + down 122.3 MB) + LM head 1054.4 MB, ctx 515",
                      2: "profiles/r2_config2_decode_ncu.md: 32 x 3321.8 MB (attention 2668.3 + merge 59.9 + gate/up 256.0 + O/down 193.2 "
                         "+ QKV 56.2 + add_rmsnorm 58.8 + swiglu 29.4) + LM head 1.06 GB, B = 512"}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    """Sustained dense bf16 TFLOP/s (the prefill GEMMs run inside a long step, B200_PROFILING.md)."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
        except Exception:  # noqa: BLE001
            pass
    return 1400.0, "fallback (B200_PROFILING.md)"


def window_cfg(w: dict) -> dict:
    """hostsim keys describing the context-window lengths of a workload"""
    if w.get("prompt_min"):
        return {"prompt_tokens_min": w["prompt_min"], "prompt_tokens_max": w["prompt_max"]}
    return {"prompt_tokens": w["prompt_tokens"]}


def window_desc(w: dict) -> str:
    return (f"windows log-uniform {w['prompt_min']}..{w['prompt_max']} tokens" if w.get("prompt_min")
            else f"windows of {w['prompt_tokens']} tokens")


def dump_outputs(out_dir: str, outputs: list, max_tokens: int) -> None:
    """status.output of every Task as UTF-8 byte rows (float32, -1 padding) in out_dir/task_output_bytes.npy"""
    import numpy as np
    rows = [o.encode() for o in outputs]
    width = max([5 * max_tokens] + [len(r) for r in rows])
    arr = np.full((len(rows), width), -1.0, dtype=np.float32)
    for i, r in enumerate(rows):
        arr[i, :len(r)] = np.frombuffer(r, dtype=np.uint8)
    assert arr.nbytes <= 64 << 20, arr.shape
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "task_output_bytes.npy"), arr)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.samples, self.proc, self.thread = [], None, None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.samples.append(parts)

    def stop(self) -> dict:
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:  # noqa: BLE001
                self.proc.kill()
        sm, mx, reasons = [], 0.0, set()
        for p in self.samples:
            try:
                sm.append(float(p[0]))
                mx = max(mx, float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def run_reference(args) -> dict:
    """CPU reconcile loop (restated) against the loopback stub server, all host cores."""
    from agentcontrolplane_b200 import host
    cores = os.cpu_count() or 1
    with host.StubServer() as srv:
        cfg = {"tasks": 2000, "workers": cores, "provider": "openai", "model": "gpt-4o", "baseURL": srv.base_url,
               "seed": 1, **window_cfg(WORKLOAD)}
        # size one step to >= ~2 s of CPU work
        cfg["tasks"] = 2000
        while True:
            t0 = time.perf_counter()
            host.hostsim_run(cfg)
            w = time.perf_counter() - t0
            if w >= 1.5 or cfg["tasks"] >= 1000000:
                break
            cfg["tasks"] = int(cfg["tasks"] * max(2.0, min(16.0, 2.5 / max(w, 1e-3))))
        for _ in range(args.warmup):
            host.hostsim_run(cfg)
        t0 = time.perf_counter()
        total, p50s = 0, []
        for i in range(args.steps):
            r = host.hostsim_run(dict(cfg, seed=i + 1))
            total += r["reconciles"]
            p50s.append(r["step_ms_p50"])
        wall = time.perf_counter() - t0
        one = host.hostsim_run(dict(cfg, workers=1, tasks=max(100, cfg["tasks"] // cores)))
    value = total / wall
    sample = f"{cfg['tasks']} Task reconciles per step, {window_desc(WORKLOAD)}, stub completion server on loopback"
    return {"impl": "reference", "metric": "task_reconciles_per_s", "value": value, "unit": "reconciles/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD["name"], "reference_path": "C++ restatement of the Go reconcile loop "
                       "(sendLLMRequest + langchaingo openai wire) doing HTTP/1.1 to a local stub completion server; "
                       "no model arithmetic happens on the reference's side of this path"},
            "p50_step_ms": sorted(p50s)[len(p50s) // 2],
            "cpu_baseline": {"value": value, "unit": "reconciles/s", "cores": cores, "kind": "port", "sample": sample,
                             "single_worker_value": one["reconciles_per_s"]},
            "e2e": {"value": value, "unit": "reconciles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def cpu_baseline_sample() -> dict:
    from agentcontrolplane_b200 import host
    cores = os.cpu_count() or 1
    with host.StubServer() as srv:
        cfg = {"tasks": 400, "workers": cores, "provider": "openai", "model": "gpt-4o", "baseURL": srv.base_url,
               "seed": 7, **window_cfg(WORKLOAD)}
        # grow the sample until it is ~10 s of CPU work (thread start-up dominates tiny samples)
        cfg["tasks"] = 2000
        while True:
            t0 = time.perf_counter()
            r = host.hostsim_run(cfg)
            wall = time.perf_counter() - t0
            if wall >= 8.0 or cfg["tasks"] >= 2000000:
                break
            cfg["tasks"] = int(cfg["tasks"] * max(2.0, min(16.0, 10.0 / max(wall, 1e-3))))
        one = host.hostsim_run(dict(cfg, workers=1, tasks=max(200, cfg["tasks"] // (2 * cores))))
    return {"value": r["reconciles"] / wall, "unit": "reconciles/s", "cores": cores, "kind": "port",
            "sample": f"{cfg['tasks']} Task reconciles ({window_desc(WORKLOAD)}) of the restated Go loop "
                      f"over HTTP to a loopback stub completion server, {wall:.1f} s",
            "single_worker_value": one["reconciles_per_s"], "p50_step_ms": r["step_ms_p50"]}


def main():
    global WORKLOAD
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default=WORKLOAD["model"])
    ap.add_argument("--layers", type=int, default=0, help="dev only: truncate depth (result is then NOT a bench value)")
    ap.add_argument("--config", type=int, default=2, choices=sorted(WORKLOADS),
                    help="BASELINE.json config index (2 = default; 1 = 64 x 512; 3 = 70B TP=8, 4 = Mixtral EP=8: ONE process on an 8-GPU box, --gpus 1)")
    ap.add_argument("--max-tokens-per-step", type=int, default=4096, help="engine knob: token rows per prefill step (4096 measured 1.3 %% faster than 8192)")
    ap.add_argument("--tp", type=int, default=0, help="dev only: override the tensor-parallel degree of --config 3")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the Task outputs of the last timed step to DIR/task_output_bytes.npy (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the outputs of --impl ours")
    WORKLOAD = dict(WORKLOADS[args.config])
    if args.config in (3, 4):
        if args.model == WORKLOADS[1]["model"]:
            args.model = WORKLOAD["model"]
        else:
            WORKLOAD["name"] += f" [DEV: model={args.model}]"
        if args.tp:
            WORKLOAD["tp"] = args.tp
            WORKLOAD["name"] += f" [DEV: tp={args.tp}]"

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    dry = None
    if WORKLOAD.get("prompt_min"):
        # mixed windows: the very windows hostsim will build (dry run, no Task reconciled); both arms
        # describe — and run — the same window distribution
        from agentcontrolplane_b200 import host as _host
        dry = _host.hostsim_run({"tasks": WORKLOAD["tasks"], "provider": "openai", "dry_run": True, **window_cfg(WORKLOAD)})
        WORKLOAD["name"] += f" [{dry['prompt_tokens_total']} window tokens per step, longest {dry['prompt_tokens_max']}]"

    if args.impl == "reference":
        if rank == 0:
            print(json.dumps(run_reference(args)), flush=True)
        return

    import torch
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from agentcontrolplane_b200 import host
    from agentcontrolplane_b200.engine import Engine

    n_tasks, plen, max_new = WORKLOAD["tasks"], WORKLOAD["prompt_tokens"], WORKLOAD["max_tokens"]
    if WORKLOAD["tools"]:
        # the synthetic tokenizer is byte-level: the agent's tool schemas render to more tokens than a BPE
        # vocabulary would need, so the window can exceed the nominal length (never less work than configured)
        probe = host.hostsim_window_tokens(plen, WORKLOAD["tools"])
        if probe != plen:
            WORKLOAD["name"] += f" [windows are {probe} tokens: tool schemas under the byte-level synthetic tokenizer]"
            plen = probe
    pages_per_seq = (plen + max_new) // 32 + 2
    if WORKLOAD["tool_loop"] or WORKLOAD.get("delegation_depth"):
        pages_per_seq += 12   # second LLM step: window + tool call + tool result
    if WORKLOAD.get("delegation_depth"):
        pages_per_seq += 16   # the delegate tool's schema in the window + the scripted delegate call (byte-level tokenizer)
        # the child's Output comes back as the ToolCall result: a generated token re-encodes to up to 5 byte tokens
        # under the synthetic vocabulary (" " + base-26 letters), so the fold-back adds up to 5 x max_tokens rows
        pages_per_seq += (5 * max_new) // 32 + 2
    kv_pages = n_tasks * pages_per_seq * 2 + 8
    if dry is not None:   # mixed windows: size the KV pool from the dry run
        pages_per_seq = (dry["prompt_tokens_max"] + max_new) // 32 + 2
        kv_pages = dry["prompt_tokens_total"] // 32 + n_tasks * (max_new // 32 + 3) + 64
    ecfg = {"model": args.model, "device": local_rank, "max_batch": max(64, n_tasks), "max_tokens_per_step": args.max_tokens_per_step,
            "kv_pages": kv_pages, "max_pages_per_seq": max(32, pages_per_seq), "tp": WORKLOAD["tp"],
            # config 1 measures cold Task steps: KV retention stays off so that no prefill work is skipped;
            # the tool loop of config 3 is exactly the case retention exists for (second turn of a Task)
            "prefix_cache": bool(WORKLOAD["tool_loop"] or WORKLOAD.get("delegation_depth"))}
    if args.layers:
        ecfg["layers"] = args.layers
    eng = Engine(ecfg)
    sim = {"tasks": n_tasks, "workers": n_tasks, "provider": "local", "model": args.model, "max_tokens": max_new,
           "tools": WORKLOAD["tools"], "tool_loop": WORKLOAD["tool_loop"],
           **(window_cfg(WORKLOAD) if WORKLOAD.get("prompt_min") else {"prompt_tokens": plen})}
    for key in ("arrival_rate", "delegation_depth"):
        if WORKLOAD.get(key):
            sim[key] = WORKLOAD[key]

    def barrier():
        torch.cuda.synchronize(local_rank)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(local_rank)

    for i in range(args.warmup):
        host.hostsim_run(dict(sim, seed=1000 + i), eng)
    eng.stats_reset()
    s0 = eng.stats()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    t0 = time.perf_counter()
    reconciles, p50s, phases, task_p50, task_p99 = 0, [], {}, [], []
    for i in range(args.steps):
        r = host.hostsim_run(dict(sim, seed=i + 1, return_outputs=bool(args.dump_outputs) and i == args.steps - 1), eng)
        reconciles += r["reconciles"]
        p50s.append(r["step_ms_p50"])
        task_p50.append(r.get("task_ms_p50"))
        task_p99.append(r.get("task_ms_p99"))
        for k, v in r["final_phases"].items():
            phases[k] = phases.get(k, 0) + v
        if r["final_phases"].get("Failed"):
            # a Failed Task is work that was NOT done (its remaining LLM steps never ran): the number would be invalid
            raise SystemExit(f"bench: {r['final_phases']['Failed']} Tasks ended Failed — {r.get('first_error')}")
    if reconciles == 0 or not phases.get("FinalAnswer"):
        raise SystemExit(f"bench: no Task reached FinalAnswer (phases {phases}) — {r.get('first_error')}")
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop() if sampler else None
    s1 = eng.stats()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r["outputs"], max_new)
    # extra key: BASELINE config 1 (64 Tasks x 512-token windows) on the same engine, outside the timed region
    config1 = None
    if args.config == 2 and rank == 0:
        w1 = WORKLOADS[1]
        sim1 = {"tasks": w1["tasks"], "workers": w1["tasks"], "provider": "local", "model": args.model,
                "max_tokens": w1["max_tokens"], "prompt_tokens": w1["prompt_tokens"], "tools": 0, "tool_loop": False}
        host.hostsim_run(dict(sim1, seed=2000), eng)
        eng.stats_reset()
        t1 = time.perf_counter()
        n1 = sum(host.hostsim_run(dict(sim1, seed=2001 + i), eng)["reconciles"] for i in range(3))
        w1_wall = time.perf_counter() - t1
        c1 = eng.stats()
        hbm_peak, _ = measured_peaks()
        tf_peak, _ = measured_tensor_peak()
        c1_dec_s, c1_pre_s = c1["decode_ms"] / 1e3, c1["prefill_ms"] / 1e3
        config1 = {"workload": w1["name"], "steps": 3,
                   "value": n1 / (c1_dec_s + c1_pre_s), "e2e": n1 / w1_wall, "unit": "reconciles/s",
                   "decode_tokens_per_s": c1["decode_tokens"] / c1_dec_s, "p50_decode_step_ms": c1.get("decode_step_ms_p50"),
                   "roofline_decode_frac": c1["decode_bytes_algorithmic"] / c1_dec_s / 1e9 / hbm_peak,
                   "roofline_prefill_frac": c1["prefill_flops_algorithmic"] / c1_pre_s / 1e12 / tf_peak,
                   "prefill_tokens_per_s": c1["prefill_tokens"] / c1_pre_s}
    dev_s = (s1["decode_ms"] + s1["prefill_ms"]) / 1e3
    from agentcontrolplane_b200.replicas import aggregate
    wall_max, dev_max, (total_reconciles, total_decode_tokens) = aggregate(
        dist, f"cuda:{local_rank}", wall, dev_s, [float(reconciles), float(s1["decode_tokens"])])
    _, dec_max, _ = aggregate(dist, f"cuda:{local_rank}", 0.0, s1["decode_ms"] / 1e3, [0.0])

    # N = 8 only: BASELINE config 3 (Llama-3-70B, tensor parallel over the 8 GPUs of ONE process, 256 Tasks
    # with the tool-call loop) measured right after the data-parallel line, so that the driver's scaling run
    # records it.  Every rank frees its GPU first; rank 0 runs `bench.py --config 3` as a SUBPROCESS (a crash
    # there costs the extra key, never the headline line); the other ranks wait on the rendezvous store
    # (host-side, no NCCL kernel spinning on their GPUs).
    tp8 = None
    # dev: ACP_BENCH_TP_WORLD=2 ACP_BENCH_TP_ARGS="--model llama-3-8b --tp 2" exercises the same flow on a 2-GPU box
    tp_world = int(os.environ.get("ACP_BENCH_TP_WORLD", "8"))
    if world == tp_world and world > 1 and args.config == 2 and not args.layers and os.environ.get("ACP_BENCH_TP8", "1") != "0":
        eng.close()
        eng = None
        barrier()
        store = torch.distributed.distributed_c10d._get_default_store()
        if rank == 0:
            try:
                env = {k: v for k, v in os.environ.items()
                       if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "LOCAL_WORLD_SIZE", "GROUP_RANK", "ROLE_RANK", "MASTER_ADDR", "MASTER_PORT",
                                    "TORCHELASTIC_RUN_ID", "CUDA_VISIBLE_DEVICES")}
                out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "3", "--steps", "2", "--warmup", "1",
                                      *os.environ.get("ACP_BENCH_TP_ARGS", "").split()],
                                     capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
                j = json.loads(out.stdout.strip().splitlines()[-1])
                tp8 = {"workload": j["config"]["workload"], "parallelism": j["config"]["parallelism"], "n_gpus": j["n_gpus"],
                       "value": j["value"], "e2e": j["e2e"]["value"], "unit": j["unit"], "steps": j["steps"],
                       "decode_tokens_per_s": j["decode_tokens_per_s"], "p50_decode_step_ms": j["p50_decode_step_ms"],
                       "p99_decode_step_ms": j.get("p99_decode_step_ms"), "roofline_decode_frac_per_gpu": j["roofline"]["frac"],
                       "roofline_prefill_frac_per_gpu": j["roofline_prefill"]["frac"], "gpu_launches": j["gpu_launches"],
                       "llm_steps_per_task": j["config"]["llm_steps_per_task"], "prefix_tokens_reused": j["config"]["prefix_tokens_reused"]}
            except Exception as e:  # noqa: BLE001
                tail = ""
                try:   # what the subprocess said last (device-side printf of a bounded wait lands on stdout)
                    tail = " | stdout: " + " / ".join(out.stdout.strip().splitlines()[-2:])[-300:] + " | stderr: " + " / ".join(out.stderr.strip().splitlines()[-3:])[-400:]
                except Exception:  # noqa: BLE001
                    pass
                tp8 = {"unavailable": (f"{type(e).__name__}: {e}"[:200] + tail)[:1000]}
            store.set("acp_bench_tp8_done", "1")
        else:
            import datetime
            store.wait(["acp_bench_tp8_done"], datetime.timedelta(seconds=1500))

    if rank == 0:
        peak, peak_src = measured_peaks()
        dec_s = s1["decode_ms"] / 1e3
        # per GPU: a tensor-parallel engine streams 1/tp of the bytes on each GPU
        achieved = s1.get("decode_bytes_algorithmic_per_gpu", s1["decode_bytes_algorithmic"]) / dec_s / 1e9 if dec_s > 0 else 0.0
        launches = s1["kernel_launches"] - s0["kernel_launches"]
        tf_peak, tf_src = measured_tensor_peak()
        pre_s = s1["prefill_ms"] / 1e3
        pre_tf = s1.get("prefill_flops_algorithmic", 0.0) / WORKLOAD["tp"] / pre_s / 1e12 if pre_s > 0 else 0.0
        line = {
            "metric": "task_reconciles_per_s", "value": total_reconciles / dev_max, "unit": "reconciles/s",
            "n_gpus": world * WORKLOAD["tp"], "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall_max / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD["name"] + (f" [DEV: layers={args.layers}]" if args.layers else ""),
                       "weights": f"seeded synthetic bf16 at {args.model} shapes (seed 0xACB200)",
                       "parallelism": (f"dp{world} (one engine replica per GPU, no collective)" if WORKLOAD["tp"] == 1 else
                                       f"tp{WORKLOAD['tp']} (one process; fused peer-memory all-reduce + residual + RMSNorm "
                                       "x2 per layer over NVLink, tp_comm.cu)"),
                       "prefix_hits": s1.get("prefix_hits", 0), "prefix_tokens_reused": s1.get("prefix_tokens_reused", 0),
                       "l2": (f"inputs larger than L2: every decode step streams {s1['decode_bytes_algorithmic'] / max(1, s1['decode_steps']) / 1e9:.1f} GB "
                              "of weights + KV (all GPUs) through a 126 MB L2 per GPU"),
                       "llm_steps_per_task": total_reconciles / (world * n_tasks * args.steps),
                       "final_phases": phases},
            "decode_tokens_per_s": total_decode_tokens / dec_max if dec_max > 0 else 0.0,  # all ranks / max decode time
            "decode_tokens_per_s_rank0": s1["decode_tokens"] / dec_s if dec_s > 0 else 0.0,
            "prefill_tokens_per_s_rank0": s1["prefill_tokens"] / (s1["prefill_ms"] / 1e3) if s1["prefill_ms"] else 0.0,
            "p50_decode_step_ms": s1.get("decode_step_ms_p50"),
            "p99_decode_step_ms": s1.get("decode_step_ms_p99"),
            "p50_reconcile_ms": sorted(p50s)[len(p50s) // 2],
            "task_ms_p50": sorted(task_p50)[len(task_p50) // 2] if task_p50 and task_p50[0] is not None else None,
            "task_ms_p99": max(task_p99) if task_p99 and task_p99[0] is not None else None,
            "e2e": {"value": total_reconciles / wall_max, "unit": "reconciles/s",
                    "h2d_bytes_per_step": (s1["h2d_bytes"] - s0["h2d_bytes"]) / args.steps,
                    "d2h_bytes_per_step": (s1["d2h_bytes"] - s0["d2h_bytes"]) / args.steps,
                    "decode_tokens_per_s": total_decode_tokens / wall_max},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         # DRAM bytes of one decode step from the committed ncu --set full capture (config 1 only)
                         "traffic": NCU_TRAFFIC.get(args.config) if not args.layers else None,
                         "traffic_source": NCU_TRAFFIC_SOURCE.get(args.config),
                         "peak_source": peak_src,
                         "kernel": "one decode step (all launches of the step, CUDA events on the engine stream)",
                         "bytes_per_decode_step": s1["decode_bytes_algorithmic"] / max(1, s1["decode_steps"]),
                         "decode_steps_timed": s1["decode_steps"],
                         "share_of_device_time": dec_s / (dec_s + pre_s) if dec_s + pre_s > 0 else None},
            # the other phase of the same timed region: prefill is dense contraction (tensor bound)
            "roofline_prefill": {"bound": "tensor", "achieved": pre_tf, "peak": tf_peak, "unit": "TFLOP/s",
                                 "frac": pre_tf / tf_peak, "traffic": None, "peak_source": tf_src,
                                 "kernel": "all prefill steps (QKV/O/gate-up/down GEMMs on tcgen05 + causal paged attention + LM head rows), "
                                           "CUDA events on the engine stream; FLOPs = 2 per layer weight per token + 4*head_dim per (query head, visible key)",
                                 "flops_per_prefill_token": s1.get("prefill_flops_algorithmic", 0.0) / max(1, s1["prefill_tokens"]),
                                 "prefill_tokens_timed": s1["prefill_tokens"],
                                 "share_of_device_time": pre_s / (dec_s + pre_s) if dec_s + pre_s > 0 else None},
            "clocks": clocks,
        }
        if config1 is not None:
            line["config1"] = config1
        if tp8 is not None:
            line["tp8_70b"] = tp8
        if world == 1 and args.config not in (3, 4):
            line["cpu_baseline"] = cpu_baseline_sample()
        print(json.dumps(line), flush=True)
    if eng is not None:
        eng.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
