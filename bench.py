#!/usr/bin/env python
"""bench.py -- decode tokens/s of the quantized forward pass (BASELINE.json metric) on N B200s.

  python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
  python bench.py --impl reference --steps K --warmup W  # the reference's CPU path (jlama-native C kernels
                                                         # + restated orchestration) on the box's host cores

Workload (config.workload): Llama-3-8B, Jlama-Q4 weights (synthetic, real dims), Q8 activations, F32 KV,
batch-1 greedy decode after a short prompt.  One "step" = one decoded token (forward(token, pos) + sample).

  value : tokens/s with the token ids resident in HBM (device-side feedback loop, CUDA-graph replays),
          timed with CUDA events on the model stream, max over ranks.
  e2e   : tokens/s through the reference-facing call -- jl_model_generate (AbstractModel.generate at temperature 0)
          with HOST token buffers: every decoded token copies token/position/session ids host->device from pinned
          memory and the sampled token back (a host round trip per step inside the timed region).
  roofline : achieved = algorithmic weight bytes per token (SURVEY 8d: 0.625 B/weight Q4 incl. f32 block scales) / the time
          of the weight-streaming kernel inside the timed region: the persistent decode kernel is the step itself (one
          launch per token, CUDA events over the timed region); for the per-op graph path the GEMV launches' summed
          durations come from device-side %globaltimer stamps inside one replayed graph (tools/ktrace.py child process).
          step_frac = the same bytes / whole-step time (the north-star "fraction of HBM roofline"); peak = MEASURED_PEAKS.json.
  --dump-outputs DIR : after the timed steps, DIR/tokens.npy holds the token id each timed step returned, as float64.  Weights
          and prompt are seeded, so two builds run with the same arguments can be compared token for token.
  cpu_baseline : the oracle driving the reference's own C kernels (oracle/_ref) on a bounded sample, with Jlama's default
          thread count (half the available CPUs); `--impl reference` uses all of them.
  config.prefill : tokens/s of a 2048-token prompt on the tcgen05 prefill path (N = 1 only).
  parity : in-run check of tokens and logits against both CPU implementations, plus their distance from each other.

Timing hygiene: W>=3 warm-up steps; weights (4.7 GB/token) are far larger than the 126 MB L2, so no L2
flush is needed ("inputs larger than L2"); clocks sampled with nvidia-smi during the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.proc, self.lines = gpu, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


_REAL_STDOUT = None


def capture_stdout():
    """Route fd 1 to stderr for the whole run (NCCL and friends print banners to stdout); the JSON line is written to
    the original stdout by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, line)
    else:
        os.write(_REAL_STDOUT, line)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic(cfg):
    """DRAM bytes (read + written) of one decode step from the committed ncu capture of the persistent decode kernel
    (profiles/r2_ncu_traffic.json: `ncu --set full`, one launch = one token), or None for another model."""
    p = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p))
    if d.get("model") != cfg["name"]:
        return None
    return int(d["per_token_bytes"])


def make_model_weights(cfg, mode, q4_fn=None):
    """Synthetic checkpoint with the real dims.  mode "quantize" (default): W ~ N(0, 0.02^2) f32 quantised with the
    reference quantiser semantics (SURVEY 8d) -- by the GPU weight quantiser (jl_quantize_q4_weights, byte-identical to
    the reference's Q4ByteBufferTensor constructor, tests/test_gpu_ops.py) in the product arm, by the oracle's C
    quantiser in the reference arm; same seeds, same bytes."""
    from jlama_b200 import native, synth
    t0 = time.time()
    w = synth.make_weights(cfg, wdtype=native.Q4, mode=mode, q4_fn=q4_fn)
    log("[bench] synthetic %s checkpoint (%s) generated in %.1fs" % (cfg["name"], mode, time.time() - t0))
    return w


def gpu_q4_quantizer(ctx):
    from jlama_b200 import native

    def q4(x):
        x = np.ascontiguousarray(x, dtype=np.float32)
        q = np.empty((x.shape[0], x.shape[1] // 2), dtype=np.uint8)
        sc = np.empty((x.shape[0], x.shape[1] // 32), dtype=np.float32)
        ctx.check(ctx.lib.jl_quantize_q4_weights(ctx.h, native.ptr(x), x.shape[0], x.shape[1], native.ptr(q), native.ptr(sc)))
        return q, sc
    return q4


def config3_workload(ctx, cfg, peak, sessions=8, prompt_tokens=2048, decode_tokens=128):
    """BASELINE config 3: Llama-3-8B Q8_0 (int8 weights + one f32 scale per 32-element block, Q8ByteBufferTensor.java:68-90),
    `sessions` concurrent sessions sharing the weights (the reference's batch: KvBufferCache.java:58-60), prefill 2048 /
    decode 128 each.  Weights: synthetic int8 bytes + scales ("direct").  Everything is driven through the host-buffer
    C ABI (jl_model_batch_forward / jl_model_decode), so both numbers are end-to-end figures."""
    from jlama_b200 import native, synth
    from jlama_b200.model import LlamaModel
    t0 = time.time()
    w8 = synth.make_weights(cfg, wdtype=native.I8, mode="direct")
    log("[bench] config 3: synthetic Q8_0 checkpoint generated in %.1fs" % (time.time() - t0))
    prompt_tokens = min(prompt_tokens, cfg["ctx"] - decode_tokens - 8)
    # prompts go through the tensor-core prefill path in one chunk each (Q8_0 blocks are dequantised into the BF16 weight tile like Q4)
    m = LlamaModel(ctx, cfg, w8, max_context=prompt_tokens + decode_tokens + 8, max_sessions=sessions, prefill_tensor_core=1,
                   max_batch=max(256, min(prompt_tokens, 2048)))
    wbytes = m.weight_bytes()
    prompts = [synth.random_prompt(cfg, prompt_tokens, seed=500 + s) for s in range(sessions)]
    for s in range(sessions):  # warm-up: kernel load and the KV pages of every session (pages stay allocated across a reset)
        m.batch_forward(prompts[s], 0, session=s)
        m.reset_session(s)
    ctx.sync()
    t0 = time.perf_counter()
    firsts = []
    for s in range(sessions):
        m.batch_forward(prompts[s], 0, session=s)
        firsts.append(m.sample(session=s, want_logits=False)[0])
    ctx.sync()
    prefill_s = time.perf_counter() - t0
    toks = np.array(firsts, dtype=np.int32)
    pos = np.full(sessions, prompt_tokens, dtype=np.int32)
    for _ in range(4):  # warm-up (captures the batch graph)
        toks, _ = m.decode(toks, pos)
        pos += 1
    ctx.sync()
    l0 = ctx.kernel_launches()
    t0 = time.perf_counter()
    n = decode_tokens - 4
    per_step = []
    for _ in range(n):
        ts = time.perf_counter()
        toks, _ = m.decode(toks, pos)  # returns after the sampled tokens are back on the host
        per_step.append(time.perf_counter() - ts)
        pos += 1
    ctx.sync()
    dt = time.perf_counter() - t0
    launches = ctx.kernel_launches() - l0
    hs = cfg["E"] // cfg["heads"]
    kv_bytes = sessions * cfg["layers"] * 2 * cfg["kv_heads"] * hs * 4 * (prompt_tokens + 4 + n / 2.0 + 1)
    step = dt / n
    out = {"workload": "%s Q8_0 (int8 weights + f32 block scales, Q8 activations, F32 KV), %d sessions, prefill %d / decode %d, direct synthetic weights"
                       % (cfg["name"], sessions, prompt_tokens, decode_tokens),
           "prefill_tokens_per_s": sessions * prompt_tokens / prefill_s, "prefill_path": "tcgen05 BF16 GEMM + tiled tensor-core attention, one 2048-token chunk per session",
           "decode_tokens_per_s": sessions / step, "decode_ms_per_step": 1e3 * step, "decode_ms_per_step_median": 1e3 * float(np.median(per_step)),
           "bytes_per_step": {"weights": wbytes, "kv": kv_bytes}, "frac_of_hbm_peak": (wbytes + kv_bytes) / 1e9 / step / peak,
           "launches_per_step": launches / n, "decode_mode": m.decode_mode(sessions),
           "timing": "host clock around the host-buffer C-ABI calls (tokens H2D, sampled tokens D2H every step)"}
    m.close()
    return out


def dump_tokens(directory, tokens):
    """--dump-outputs: the token ids the timed steps returned (float64 holds them exactly)."""
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "tokens.npy"), np.asarray(tokens, dtype=np.float64))


def teacher_forced_logits(model, prompt, ref_tokens):
    """Feed the GPU the REFERENCE's tokens (every rank of a tensor-parallel job runs this with the same tokens): logits per step."""
    n = len(ref_tokens)
    model.reset_session(0)
    model.batch_forward(prompt, 0)
    _, lg = model.sample(want_logits=True)
    logits = [lg]
    for i in range(1, n):
        _, lg = model.decode(np.array([ref_tokens[i - 1]], dtype=np.int32), np.array([len(prompt) + i - 1], dtype=np.int32), want_logits=True)
        logits.append(lg[0])
    return logits


def teacher_forced_parity(logits, ref_logits):
    """Every step compares the two sides on identical inputs (a free-running comparison stops being meaningful at the first
    divergent token).  Where the arg-max differs, `reference_gap_rel` says how much the reference itself prefers its token over
    the GPU's (relative to the largest |logit|): on the synthetic random-weight network many steps are near ties -- the
    reference's AVX-512 kernels and the plain-C port of the same arithmetic pick different tokens at step 0 of the bench prompt
    (tools/parity_margin.py, profiles/r2_parity_margin.txt)."""
    n = len(ref_logits)
    rels, agree, dis = [], 0, []
    for i in range(n):
        rl = np.asarray(ref_logits[i])
        mx = float(np.abs(rl).max())
        rel = float(np.abs(logits[i] - rl).max() / mx)
        rels.append(rel)
        gt, rt = int(np.argmax(logits[i])), int(np.argmax(rl))
        if gt == rt:
            agree += 1
        else:
            dis.append({"step": i, "reference_gap_rel": float((rl[rt] - rl[gt]) / mx), "logit_rel_err": rel})
    return {"steps": n, "argmax_agree": agree, "max_logit_rel_err": max(rels), "median_logit_rel_err": float(np.median(rels)),
            "disagreements": dis[:8], "all_disagreements_are_near_ties": all(d["reference_gap_rel"] <= d["logit_rel_err"] for d in dis)}


def first_divergence(a, b):
    for i, (x, y) in enumerate(zip(a, b)):
        if int(x) != int(y):
            return i
    return None


def cpu_reference_decode(cfg, weights, prompt, n_new, threads=None):
    """Reference-equivalent CPU path: restated orchestration + the reference's own C kernels (oracle/_ref)."""
    from oracle import oracle as o
    label = o.load_reference_kernels()
    o.use_reference_kernels(label is not None)
    # the reference's default executor: max(2, availableProcessors/2) threads (PhysicalCoreExecutor.java:27)
    o.set_num_threads(threads or max(2, o.available_cpus() // 2))
    m = o.OracleLlama(cfg, weights, act_q8=True)
    m.reset()
    t0 = time.time()
    hidden = m.batch_forward(prompt, 0)
    tok, logits0 = m.sample(hidden)
    t1 = time.time()
    toks, step_logits = [tok], [logits0]
    for i in range(1, n_new):
        hidden = m.batch_forward([toks[-1]], len(prompt) + i - 1)
        tok, lg = m.sample(hidden)
        toks.append(tok)
        step_logits.append(lg)
    t2 = time.time()
    m.close()
    return dict(tokens=toks, logits=step_logits, prefill_s=t1 - t0, decode_s=t2 - t1, kind="reference" if label else "port",
                label=label or "plain-C restatement (oracle/jlama_oracle.c)", threads=o.num_threads())


def run_reference_arm(args):
    from jlama_b200 import synth
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = synth.get_config(args.model)
    from oracle import oracle as o
    w = make_model_weights(cfg, args.weights, q4_fn=o.quantize_q4)
    prompt = synth.random_prompt(cfg, args.prompt)
    n = args.warmup + args.steps
    label = o.load_reference_kernels()
    o.use_reference_kernels(label is not None)
    # "all the host threads it can use", capped where more threads stop helping a bandwidth-bound GEMV
    o.set_num_threads(args.cpu_threads or min(o.available_cpus(), 64))
    log("[bench] reference arm: %s, %d threads (of %d available CPUs)" % (label, o.num_threads(), o.available_cpus()))
    m = o.OracleLlama(cfg, w, act_q8=True)
    m.reset()
    hidden = m.batch_forward(prompt, 0)
    tok, _ = m.sample(hidden)
    pos = len(prompt)
    for _ in range(args.warmup):
        hidden = m.batch_forward([tok], pos)
        tok, _ = m.sample(hidden)
        pos += 1
    t0 = time.time()
    toks = []
    for _ in range(args.steps):
        hidden = m.batch_forward([tok], pos)
        tok, _ = m.sample(hidden)
        toks.append(tok)
        pos += 1
    dt = time.time() - t0
    if args.dump_outputs:
        dump_tokens(args.dump_outputs, toks)
    val = args.steps / dt
    cores = o.num_threads()
    out = {
        "impl": "reference", "metric": "decode tokens/s", "value": val, "unit": "tokens/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "int8xint4->f32", "data": "synthetic",
        "config": {"workload": "%s JQ4, batch=1 greedy decode after %d-token prompt (CPU: %s, %d threads)" % (
            cfg["name"], args.prompt, label or "plain-C restatement", cores), "parallelism": "cpu"},
        "cpu_baseline": {"value": val, "unit": "tokens/s", "cores": cores, "kind": "reference" if label else "port",
                         "sample": "%d decode steps after a %d-token prompt" % (args.steps, args.prompt)},
        "e2e": {"value": val, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="llama-3-8b")
    ap.add_argument("--weights", default="quantize", choices=["direct", "quantize"])
    ap.add_argument("--prompt", type=int, default=32)
    ap.add_argument("--cpu-tokens", type=int, default=33, help="tokens generated by the cpu_baseline / parity sample (1 + decode steps)")
    ap.add_argument("--prefill-tokens", type=int, default=2048, help="prompt length of the tensor-core prefill measurement (0 = skip)")
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parity-port-tokens", type=int, default=0, help="tokens also checked against the plain-C oracle port (slow; off by default)")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-config3", action="store_true", help="skip the BASELINE config-3 measurement (8B Q8_0, 8 sessions, prefill 2048 / decode 128)")
    ap.add_argument("--no-persistent", action="store_true", help="decode through the CUDA graph of per-op kernels instead of the persistent kernel")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the token ids of the timed steps to DIR/tokens.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    capture_stdout()

    if args.impl == "reference":
        return run_reference_arm(args)

    from jlama_b200 import native, synth
    from jlama_b200.model import LlamaModel

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        log("[bench] WORLD_SIZE=%d but --gpus %d; using WORLD_SIZE" % (world, args.gpus))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl")

    cfg = synth.get_config(args.model)
    ctx = native.Context(local_rank)
    if world > 1:
        import torch
        idbuf = np.zeros(128, dtype=np.uint8)
        if rank == 0:
            ctx.check(ctx.lib.jl_comm_unique_id(ctx.h, native.ptr(idbuf)))
        t = torch.from_numpy(idbuf).cuda()
        dist.broadcast(t, 0)
        idbuf = t.cpu().numpy()
        ctx.check(ctx.lib.jl_comm_init(ctx.h, native.ptr(idbuf), rank, world))

    moe = bool(cfg.get("experts"))
    if moe and not args.no_cpu_baseline:
        log("[bench] %s: CPU baseline / in-run parity skipped (the CPU side would need the whole checkpoint in host memory; "
            "expert-parallel parity is tests/test_gpu_tp.py)" % cfg["name"])
        args.no_cpu_baseline = True
    if moe:
        # Mixtral (BASELINE config 5): experts are held whole, one rank each (e % N); every rank generates only its own tensors
        weights = synth.lazy_weights(cfg, wdtype=native.Q4, mode=args.weights, q4_fn=gpu_q4_quantizer(ctx))
    else:
        weights = make_model_weights(cfg, args.weights, q4_fn=gpu_q4_quantizer(ctx))
    prompt = synth.random_prompt(cfg, args.prompt)
    n_total = args.prompt + 2 * (args.warmup + args.steps) + 64
    t0 = time.time()
    model = LlamaModel(ctx, cfg, weights, max_context=min(cfg["ctx"], max(512, n_total)), tp_rank=rank, tp_size=world,
                       flags=native.MODEL_NO_PERSISTENT if args.no_persistent else 0)
    log("[bench] rank %d: weights uploaded in %.1fs (%.3f GB streamed per token on this rank)" % (
        rank, time.time() - t0, model.weight_bytes() / 1e9))

    def barrier():
        ctx.sync()
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- prefill + parity reference tokens -------------------------------------------------------------
    model.reset_session(0)
    barrier()
    t0 = time.time()
    model.batch_forward(prompt, 0)
    first, _ = model.sample(want_logits=False)
    ctx.sync()
    prefill_s = max_over_ranks(time.time() - t0)

    # ---- value: resident decode loop (CUDA graph replays, token ids stay in HBM) --------------------------
    pos = len(prompt)
    launches0 = ctx.kernel_launches()
    warm = model.decode_resident(first, pos, args.warmup)
    pos += args.warmup
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.15)
    l0 = ctx.kernel_launches()
    toks = model.decode_resident(int(warm[-1]), pos, args.steps)
    total_ms, _ = model.last_timing()
    barrier()
    launches = ctx.kernel_launches() - l0
    total_ms = max_over_ranks(total_ms)
    pos += args.steps
    value = args.steps / (total_ms / 1000.0)

    # ---- e2e: the reference-facing call -- generate() (AbstractModel.generate at temperature 0) through the C ABI with
    # HOST token buffers; every decoded token makes a host round trip (token/position/session ids H2D from pinned
    # memory, sampled token D2H) inside the timed region, which is the library's own decode-phase timer -------------
    barrier()
    gen_tokens, _ = model.generate(prompt, args.warmup + 1)  # warm-up (also re-captures nothing: graphs are cached)
    barrier()
    gen_tokens, _ = model.generate(prompt, args.steps + 1)
    e2e_s = max_over_ranks(model.last_timings_ms[1] / 1e3)
    e2e_prefill_s = max_over_ranks(model.last_timings_ms[0] / 1e3)
    barrier()
    clocks = sampler.stop()
    e2e = args.steps / e2e_s

    peak, peak_src = measured_peaks()
    wbytes = model.weight_bytes()
    result = {
        "metric": "decode tokens/s", "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int8xint4->f32", "data": "synthetic",
        "config": {"workload": "%s JQ4 (Q4 weights + f32 block scales, Q8 activations, F32 KV), batch=1 greedy decode, "
                               "%d-token prompt, %s synthetic weights" % (cfg["name"], args.prompt, args.weights),
                   "parallelism": ("tp%d attention + ep%d experts (expert e on rank e %% %d)" % (world, world, world) if moe else "tp%d" % world) if world > 1 else "single-gpu",
                   "l2": "inputs larger than L2 (%.2f GB of weights per token per rank vs 126 MB L2)" % (wbytes / 1e9),
                   "prompt_prefill_tokens_per_s": args.prompt / prefill_s},
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": "tokens/s", "h2d_bytes_per_step": 12, "d2h_bytes_per_step": 4},
        "gpu_launches": int(launches),
    }

    # ---- roofline of the dominant kernel -------------------------------------------------------------------------------
    # step_frac: algorithmic weight bytes of one token / the whole event-timed step (the north-star number).
    # frac: the same bytes / the time the weight-streaming kernel(s) actually ran inside the step -- for the persistent
    # decode kernel that IS the step (one launch per token); for the graph of per-op kernels it is the summed
    # (last CTA end - first CTA start) of the GEMV launches inside one replayed graph from device-side %globaltimer
    # stamps (tools/ktrace.py in a child process).  Never an eager per-launch event sum (VERDICT r1 weak #5).
    mode = model.decode_mode(1)
    step_ms = total_ms / args.steps
    step_frac = (wbytes / 1e9) / (step_ms / 1e3) / peak
    mode_name = {3: "persistent decode kernel (one cooperative launch per token)", 2: "persistent megakernel (round 1)",
                 1: "cuda graph of per-op kernels", 0: "eager"}.get(mode, str(mode))
    result["config"]["decode_mode"] = mode_name
    result["roofline"] = {"bound": "hbm", "achieved": step_frac * peak, "peak": peak, "unit": "GB/s", "frac": step_frac,
                          "traffic": measured_traffic(cfg) if world == 1 else None, "peak_source": peak_src, "step_frac": step_frac,
                          "bytes_per_token": wbytes, "us_per_token": 1000.0 * step_ms,
                          "kernel": "pdecode_kernel (all weight GEMVs, attention, lm_head + argmax of one token)" if mode >= 2 else
                                    "gemv_decode_kernel x4 per layer + lm_head gemv_kernel",
                          "method": "algorithmic bytes per token / CUDA-event time of the timed region / steps"}

    # ---- prefill throughput (BASELINE config 3 shape: 2048-token prompt) and a long-context decode point ----------------
    if world == 1 and args.prefill_tokens > 0 and not moe:
        model.close()
        ptoks = min(args.prefill_tokens, cfg["ctx"] - 72)
        # the prompt goes through in one chunk (the reference's batch size is a knob: AbstractModel.java:295-312 takes it from the caller)
        pm = LlamaModel(ctx, cfg, weights, max_context=ptoks + 72, prefill_tensor_core=1, max_batch=min(ptoks, 2048))
        long_prompt = synth.random_prompt(cfg, ptoks, seed=99)
        pm.reset_session(0)
        pm.batch_forward(long_prompt, 0)  # warm-up (allocates the KV pages of the whole prompt)
        pm.reset_session(0)
        ctx.sync()
        t0 = time.perf_counter()
        pm.batch_forward(long_prompt, 0)
        ctx.sync()
        dt = time.perf_counter() - t0
        flops = 2.0 * (synth.linear_weight_count(cfg) - cfg["vocab"] * cfg["E"]) * ptoks
        result["config"]["prefill"] = {"tokens": ptoks, "tokens_per_s": ptoks / dt, "path": "tcgen05 BF16 GEMM (Q4 dequant fused into the smem fill, activation tiles by TMA) + tiled BF16 tensor-core attention over the pages", "chunk_tokens": min(ptoks, 2048),
                                       "linear_tflops": flops / dt / 1e12}
        # decode at position ~ptoks: the KV read (SURVEY 8d: layers * 2 * kvLength * 4 B * (p+1), F32 KV) joins the numerator
        lf, _ = pm.sample(want_logits=False)
        pm.decode_resident(lf, ptoks, 8)
        nlong = 32
        pm.decode_resident(lf, ptoks + 8, nlong)
        lms, _ = pm.last_timing()
        hs = cfg["E"] // cfg["heads"]
        kv_bytes = cfg["layers"] * 2 * cfg["kv_heads"] * hs * 4 * (ptoks + 8 + nlong / 2.0 + 1)
        lstep = lms / nlong / 1e3
        result["config"]["decode_long_context"] = {
            "position": ptoks + 8, "tokens_per_s": 1.0 / lstep, "ms_per_step": 1e3 * lstep, "kv_bytes_per_token": kv_bytes,
            "frac_of_hbm_peak_weights_plus_kv": (wbytes + kv_bytes) / 1e9 / lstep / peak}
        pm.close()
        if not args.no_config3 and cfg["name"].startswith("llama-3-8b"):
            try:
                result["config"]["config3_q8_batch8"] = config3_workload(ctx, cfg, peak)
            except Exception as e:  # noqa: BLE001 -- a secondary measurement must never break the bench line
                log("[bench] config 3 skipped: %r" % (e,))
        model = LlamaModel(ctx, cfg, weights, max_context=min(cfg["ctx"], max(512, n_total)))

    # ---- cpu_baseline + in-run parity ----------------------------------------------------------------------------------
    # N = 1: the GPU generates 1 + 32 tokens after the 32-token prompt and is compared with the reference-equivalent CPU
    # path (reference C kernels under the restated orchestration) on the same prompt; logits are compared up to and
    # including the first divergent token (afterwards the two sides see different inputs).
    # N > 1: rank 0 runs OracleLlama(tp=N) -- shard-wise partial sums added in rank order -- on a shorter sample.
    if not args.no_cpu_baseline:
        n_cpu = max(2, args.cpu_tokens if world == 1 else min(args.cpu_tokens, 9))
        cp = prompt if world == 1 else prompt[:min(len(prompt), 8)]
        r = None
        if rank == 0:
            if world == 1:
                r = cpu_reference_decode(cfg, weights, cp, n_cpu, threads=args.cpu_threads or None)
            else:
                from oracle import oracle as o
                label = o.load_reference_kernels()
                o.use_reference_kernels(label is not None)
                o.set_num_threads(args.cpu_threads or o.available_cpus())
                om = o.OracleLlama(cfg, weights, act_q8=True, tp=world)
                t0 = time.time()
                pt, pl = om.generate(cp, n_cpu)
                om.close()
                r = dict(tokens=list(pt), logits=pl, label="OracleLlama(tp=%d), %s" % (world, label or "plain-C port"),
                         decode_s=time.time() - t0, threads=o.num_threads())
        barrier()
        gt, gl = model.generate(cp, n_cpu, want_logits=True)
        ref_tokens = [int(t) for t in r["tokens"]] if rank == 0 else [0] * n_cpu
        if dist is not None:  # every rank replays the reference's tokens
            import torch
            tt = torch.tensor(ref_tokens, dtype=torch.int64, device="cuda")
            dist.broadcast(tt, 0)
            ref_tokens = [int(x) for x in tt.cpu().tolist()]
        tf_logits = teacher_forced_logits(model, cp, ref_tokens)
        if rank == 0:
            tf = teacher_forced_parity(tf_logits, r["logits"])
            div = first_divergence(gt, r["tokens"])
            upto = n_cpu if div is None else div + 1
            rel = max(float(np.abs(gl[i] - r["logits"][i]).max() / np.abs(r["logits"][i]).max()) for i in range(upto))
            div_gap = None
            if div is not None:  # how decisive was the reference's own choice at the step where the two sides part?
                rl = np.asarray(r["logits"][div])
                div_gap = float((rl[int(r["tokens"][div])] - rl[int(gt[div])]) / np.abs(rl).max())
            if world == 1:
                result["cpu_baseline"] = {"value": (n_cpu - 1) / r["decode_s"], "unit": "tokens/s", "cores": r["threads"], "kind": r["kind"],
                                          "sample": "%d decode steps after a %d-token prompt, %s" % (n_cpu - 1, len(cp), r["label"]),
                                          "prefill_tokens_per_s": len(cp) / r["prefill_s"]}
            result["parity"] = {"tokens_equal": div is None, "tokens_compared": n_cpu, "tokens_equal_count": n_cpu if div is None else div,
                                "first_divergent_position": div, "reference_gap_rel_at_divergence": div_gap, "max_logit_rel_err": rel,
                                "logits_compared_steps": upto,
                                "tolerance": 1e-2, "against": r["label"], "prompt_tokens": len(cp), "weights": args.weights,
                                "teacher_forced": tf,
                                "note": "logits of a 32-layer network with a Q8 re-quantisation in front of every projection: a 1-ulp "
                                        "summation-order difference flips single int8 activations (each ~1e-3 of a layer output, "
                                        "tests/test_gpu_layer8b.py shows the mechanism layer by layer at these shapes with 2e-7 "
                                        "agreement on flip-free steps).  The synthetic random-weight network has near-tied top "
                                        "logits: at step 0 of this prompt the reference's own top-2 gap is 4.3e-3 of max|logit| and its "
                                        "AVX-512 kernels and the plain-C port of the same arithmetic already pick different tokens "
                                        "(profiles/r2_parity_margin.txt), so free-running token equality is decided by ties; "
                                        "`teacher_forced` compares every step on the reference's own tokens and reports, for each "
                                        "arg-max disagreement, how small the reference's own preference was"}
            if world == 1 and args.parity_port_tokens > 0:
                from oracle import oracle as o
                o.use_reference_kernels(False)
                om = o.OracleLlama(cfg, weights, act_q8=True)
                n_p = args.parity_port_tokens
                pt, pl = om.generate(cp, n_p)
                om.close()
                relp = max(float(np.abs(gl[i] - pl[i]).max() / np.abs(pl[i]).max()) for i in range(n_p))
                result["parity"]["vs_plain_c_port"] = {"tokens_equal": [int(a) for a in gt[:n_p]] == [int(b) for b in pt],
                                                       "max_logit_rel_err": relp, "tokens": n_p}
                # yardstick: how far the two CPU implementations of the same arithmetic are from each other on this network
                relc = max(float(np.abs(np.asarray(r["logits"][i]) - pl[i]).max() / np.abs(pl[i]).max()) for i in range(n_p))
                result["parity"]["cpu_reference_kernels_vs_plain_c_port"] = relc
                result["parity"]["note"] = ("single-layer teacher-forced parity at the 8B shapes is in tests/test_gpu_layer8b.py; "
                                            "cpu_reference_kernels_vs_plain_c_port is the distance between two CPU implementations of "
                                            "the same arithmetic on this 32-layer network (summation order only)")
    model.close()
    if rank == 0 and world == 1 and not args.no_roofline and mode == 1:
        try:
            r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ktrace.py"), "--json", "--model", args.model],
                               cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=240)
            lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            if r.returncode == 0 and lines:
                t = json.loads(lines[-1])
                ach = wbytes / 1e9 / (t["gemv_us"] * 1e-6)
                result["roofline"].update({
                    "achieved": ach, "frac": ach / peak, "gemv_us_per_token": t["gemv_us"], "attention_us_per_token": t["attention_us"],
                    "timeline_step_ms": t["step_ms_events"], "position": t["position"],
                    "method": "algorithmic bytes / sum of per-launch (last CTA end - first CTA start) of the GEMV launches inside one "
                              "replayed decode graph, %globaltimer stamps (tools/ktrace.py); stamps add ~1% to the step"})
        except Exception as e:  # noqa: BLE001 -- diagnostics must never break the bench line
            log("[bench] in-graph timeline skipped: %r" % (e,))
    if rank == 0:
        if args.dump_outputs:
            dump_tokens(args.dump_outputs, toks)
        emit(result)
    if dist is not None:
        dist.barrier()
        ctx.lib.jl_comm_destroy(ctx.h)
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
