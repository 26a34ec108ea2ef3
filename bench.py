#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native generate path.

Workload (BASELINE.json configs[1], "C2"): Qwen2-VL-2B bf16, 1 synthetic image
336x336 (144 merged image tokens), 128 text-side prompt tokens (T = 272),
512 generated tokens, batch 1, greedy, EOS ignored; seeded random-init weights
(no checkpoints offline).  One "step" = one whole request: ViT -> merge ->
prefill -> 512 decode steps.

  python bench.py --gpus N --steps K --warmup W            # this framework
  python bench.py --impl reference ...                      # CPU restatement of the
        reference path (oracle port; mlx itself is not installable offline)
  python bench.py ... --dump-outputs DIR                    # + what the timed legs returned

Prints ONE JSON line (rank 0).  `value` = decode tokens/s with inputs resident in
HBM (CUDA events, max over ranks); `e2e` = the same request through the public
API `generate(model, processor, prompt, image)` with a HOST image (preprocessing,
pinned H2D of pixel_values, per-token D2H inside the timed region).  Every leg
times exactly K steps (C5: K runs of the whole request set).

--dump-outputs DIR (rank 0) writes, after each leg's timed steps, what its last
timed step returned to its caller as DIR/<leg>_<name>.npy: float32 for floating
point outputs (bf16 converts exactly), float64 for token ids.  Inputs and weights
are seeded, so two builds run with the same arguments can be compared file by file.
The GEMM configurations are picked by timing them at first use, and a different
split of the K sum rounds differently (seen once in the C4 prefill on a B200 at
1000 W: logits 3.5e-2 relative L2 apart between two runs of one build);
B200_WT_TUNE=0 fixes them.
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

N_TEXT, N_OUT, IMG_HW = 128, 512, (336, 336)
W_BYTES_2B = 3_087_428_608      # SURVEY §8(d): decode weight bytes / token (bf16, tied head)
KV_BYTES_PER_POS = 28_672       # 2 (k,v) * 2 kv heads * 128 * 2 B * 28 layers
DUMP_MAX_ELEMS = 1 << 20        # larger outputs are dumped as a fixed, seeded sample (all dumps stay < 64 MB)


def dump_output(dump_dir, name, x):
    """Write one output of a timed step as <dump_dir>/<name>.npy (--dump-outputs).
    Floating point -> float32, integers (token ids) -> float64, both exact.  An output of more than
    DUMP_MAX_ELEMS elements is flattened and sampled at positions fixed by its size and a constant seed."""
    import numpy as np
    import torch
    if isinstance(x, torch.Tensor):
        if x.is_cuda:
            torch.cuda.synchronize(x.device)      # device outputs are written on the engine's stream
        x = x.detach().cpu()
        x = (x.float() if x.is_floating_point() else x).numpy()
    x = np.asarray(x)
    x = x.astype(np.float32 if np.issubdtype(x.dtype, np.floating) else np.float64)
    if x.size > DUMP_MAX_ELEMS:
        pick = np.random.default_rng(0).choice(x.size, DUMP_MAX_ELEMS, replace=False)
        x = x.reshape(-1)[np.sort(pick)]
    np.save(os.path.join(dump_dir, name + ".npy"), x)


def _token_log(eng, n):
    """the last `n` token ids the engine's greedy sampler wrote (prefill's first token + decode steps)"""
    import torch
    host = torch.empty(n, dtype=torch.int32).pin_memory()
    eng.fetch_tokens(eng.tokens_launched - n, n, host)
    eng.stream.synchronize()
    return host


# ViT + merge + LM prefill FLOPs of one C2 request (SURVEY §8d: 2*M*N*K per GEMM, 4*N^2*D attention)
VIT_GFLOP, PREFILL_GFLOP_T272 = 790.7, 720.0


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _tensor_peak():
    """bf16 tensor peak for a kernel timed INSIDE a long step: the sustained cuBLAS figure."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    return 1400.0, "fallback (B200_PROFILING.md ~1.4 PFLOP/s sustained)"


def _ncu_traffic():
    """dram bytes (read + write) of ONE decode-kernel launch from the committed ncu capture
    (profiles/decode_traffic.json: written by tools/ncu_traffic.py from an `ncu --set full` run)."""
    p = os.path.join(ROOT, "profiles", "decode_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("dram_bytes"), d.get("source", "profiles/decode_traffic.json")
    return None, "no ncu capture committed"


def _cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.lower().startswith("model name"):
                    name = ln.split(":", 1)[1].strip()
                    break
            else:
                name = "unknown"
        return f"{name} ({os.cpu_count()} logical CPUs)"
    except Exception:
        return "unknown"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


def _engine_weights_to_oracle(model, cfg_o):
    """Unpack the engine's packed device weights into the oracle's name space (fp32 CPU)."""
    import torch
    w = model.engine.weights
    t, v = cfg_o.text, cfg_o.vision
    H, hd = t.hidden_size, t.hidden_size // t.num_attention_heads
    kvd = t.num_key_value_heads * hd
    out = {}

    def f(x):
        return x.detach().float().cpu()

    out["vision_tower.patch_embed.proj.weight"] = f(w["v.patch_embed.w"])
    pairs = (("norm1.weight", "ln1.w"), ("norm1.bias", "ln1.b"), ("norm2.weight", "ln2.w"),
             ("norm2.bias", "ln2.b"), ("attn.qkv.weight", "qkv.w"), ("attn.qkv.bias", "qkv.b"),
             ("attn.proj.weight", "proj.w"), ("attn.proj.bias", "proj.b"),
             ("mlp.fc1.weight", "fc1.w"), ("mlp.fc1.bias", "fc1.b"),
             ("mlp.fc2.weight", "fc2.w"), ("mlp.fc2.bias", "fc2.b"))
    for i in range(v.depth):
        for a, b in pairs:
            out[f"vision_tower.blocks.{i}.{a}"] = f(w[f"v.blk.{i}.{b}"])
    for a, b in (("ln_q.weight", "ln.w"), ("ln_q.bias", "ln.b"), ("mlp.0.weight", "fc1.w"),
                 ("mlp.0.bias", "fc1.b"), ("mlp.2.weight", "fc2.w"), ("mlp.2.bias", "fc2.b")):
        out["vision_tower.merger." + a] = f(w["v.merger." + b])
    out["language_model.model.embed_tokens.weight"] = f(w["lm.embed"])
    out["language_model.model.norm.weight"] = f(w["lm.norm"])
    for i in range(t.num_hidden_layers):
        p = f"language_model.model.layers.{i}."
        wqkv, bqkv, wgu = f(w[f"lm.{i}.wqkv"]), f(w[f"lm.{i}.bqkv"]), f(w[f"lm.{i}.wgu"])
        out[p + "input_layernorm.weight"] = f(w[f"lm.{i}.ln1"])
        out[p + "post_attention_layernorm.weight"] = f(w[f"lm.{i}.ln2"])
        out[p + "self_attn.q_proj.weight"], out[p + "self_attn.k_proj.weight"], \
            out[p + "self_attn.v_proj.weight"] = wqkv[:H], wqkv[H:H + kvd], wqkv[H + kvd:]
        out[p + "self_attn.q_proj.bias"], out[p + "self_attn.k_proj.bias"], \
            out[p + "self_attn.v_proj.bias"] = bqkv[:H], bqkv[H:H + kvd], bqkv[H + kvd:]
        out[p + "self_attn.o_proj.weight"] = f(w[f"lm.{i}.wo"])
        out[p + "mlp.gate_proj.weight"], out[p + "mlp.up_proj.weight"] = \
            wgu[:t.intermediate_size], wgu[t.intermediate_size:]
        out[p + "mlp.down_proj.weight"] = f(w[f"lm.{i}.wd"])
    return out


def cpu_reference_run(W, n_decode, threads=None):
    """Time the oracle (CPU restatement of the reference's path) on the C2 prompt:
    ViT + merge + prefill once, then `n_decode` decode steps.  Returns dict."""
    import numpy as np
    import torch
    from oracle import qwen2vl as O
    # one thread per PHYSICAL core (torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm
    # runs on rank 0 alone, so it takes the whole host.  Measured: 64 threads 3.5-4.7 tok/s, the
    # 128 logical CPUs 0.13 tok/s — hyper-thread oversubscription)
    if not threads:
        try:
            import psutil
            threads = psutil.cpu_count(logical=False)
        except Exception:
            threads = None
        threads = threads or max(1, (os.cpu_count() or 2) // 2)
        try:
            threads = min(threads, len(os.sched_getaffinity(0)))
        except Exception:
            pass
    torch.set_num_threads(threads)
    c = O.qwen2_vl_2b()
    req = O.synthetic_request(c, N_TEXT, image_hw=IMG_HW, seed=0)
    ids, pv, grid = req["input_ids"], req["pixel_values"], req["image_grid_thw"]
    R = O.Rounder("bf16")
    t0 = time.perf_counter()
    embeds, feats, pos, deltas = O.get_input_embeddings(c, W, ids, pv, grid, R)
    cache = [O.OracleKVCache() for _ in range(c.text.num_hidden_layers)]
    hidden = O.lm_layers_forward(c, W, embeds, pos, cache, R)
    logits = O.lm_head(c, W, hidden[:, -1, :], R)
    t1 = time.perf_counter()
    for _ in range(n_decode):
        lp = O.logprobs_from_logits(R, logits)
        y = O.S.argmax_lowest(lp)
        e = W["language_model.model.embed_tokens.weight"][y][:, None, :]
        p = O.decode_position_ids(cache[0].offset, deltas, 1)
        hidden = O.lm_layers_forward(c, W, e, p, cache, R)
        logits = O.lm_head(c, W, hidden[:, -1, :], R)
    t2 = time.perf_counter()
    return {"prefill_s": t1 - t0, "decode_s": t2 - t1, "n_decode": n_decode,
            "decode_tps": n_decode / (t2 - t1), "img_tps": 144 / (t1 - t0),
            "cores": torch.get_num_threads()}


W_BYTES_7B = 2 * 7_070_619_136          # SURVEY §8(d): Qwen2-VL-7B LM weights (untied head), bf16
KV_BYTES_PER_POS_7B = 57_344            # 2 * 4 kv heads * 128 * 2 B * 28 layers


def lockstep_2b(world, rank, dev, args, model, processor, ids, pvd, grid):
    """The C2 model (Qwen2-VL-2B, already resident) with `rows` copies of the C2 request as lock-step rows of one
    weight stream per GPU: what continuous batching buys on the small model (512 tokens out per row)."""
    import torch
    import torch.distributed as dist
    from mlx_vlm_b200.generate_batch import BatchGenerator
    rows, n_out = args.c5_rows, N_OUT
    eng = model.engine
    prompt = ids.reshape(-1).tolist()
    kw = {"pixel_values": pvd, "image_grid_thw": grid}

    def run():
        g = BatchGenerator(model, processor, max_tokens=n_out, completion_batch_size=rows, prefill_batch_size=rows,
                           decode_slice=32)
        uids = g.insert([prompt] * rows, [n_out] * rows, [dict(kw) for _ in range(rows)])
        toks = {u: [] for u in uids}
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        while g.has_work:
            for r in g.next()[1]:
                toks[r.uid].append(r.token)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, [toks[u] for u in uids]

    run()
    dt = 0.0
    for _ in range(args.steps):
        t, toks = run()
        dt += t / args.steps
    assert all(len(t) == n_out for t in toks)
    if args.dump_outputs:
        dump_output(args.dump_outputs, "c5_2b_rows_tokens", toks)
    step_ms = eng.last_decode_ms()
    t = torch.tensor([dt, step_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt, step_ms = t.tolist()
    peak, peak_src = _peaks()
    bytes_step = W_BYTES_2B + rows * KV_BYTES_PER_POS * (N_TEXT + 144 + n_out / 2)
    return {"workload": f"Qwen2-VL-2B, {rows} lock-step rows per GPU (the C2 request x {rows}), {n_out} tokens out each, "
                        f"admission + prefill of the rows inside the timed region, seconds = mean of {args.steps} runs",
            "rows_per_gpu": rows, "seconds": dt, "tokens_per_s": world * rows * n_out / dt,
            "decode_ms_per_step": step_ms,
            "roofline": {"bound": "hbm", "achieved": bytes_step / (step_ms / 1e3) / 1e9 if step_ms > 0 else None,
                         "peak": peak, "unit": "GB/s", "peak_source": peak_src,
                         "frac": bytes_step / (step_ms / 1e3) / 1e9 / peak if step_ms > 0 else None,
                         "algorithmic_bytes_per_step": bytes_step}}


def c5_leg(world, rank, dev, args):
    """BASELINE config 5: Qwen2-VL-7B, `rows` concurrent image+prompt requests PER GPU (64 over 8 GPUs),
    routed by parallel.generate_sharded (request i -> rank i mod N), each replica running its own
    lock-step BatchGenerator; 336x336 image, 128 text tokens in, 512 out, greedy, EOS ignored.
    Timed: max over ranks of (insert -> last token), CUDA-synchronised wall clock (host admission and
    prefill are part of serving) + the device time of the decode steps."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from mlx_vlm_b200.generate_batch import BatchGenerator
    from mlx_vlm_b200.parallel import broadcast_packed, generate_sharded, shard_requests
    from mlx_vlm_b200.utils import load_synthetic, prepare_inputs
    rows, n_out = args.c5_rows, args.c5_out
    model, proc = load_synthetic("qwen2-vl-7b", seed=1, device=dev, n_text_tokens=N_TEXT)
    model.config.eos_token_id = []
    eng = model.engine
    bc = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        tb = time.perf_counter()
        nb = broadcast_packed(model.packed_weights, src=0)
        torch.cuda.synchronize()
        bc = {"bytes": nb, "seconds": time.perf_counter() - tb}
        bc["GB_per_s"] = nb / bc["seconds"] / 1e9
    n_req = rows * world
    rng = np.random.default_rng(7)
    prompts, kws = [None] * n_req, [{} for _ in range(n_req)]
    for i in shard_requests(n_req, world, rank):       # only the router's share is prepared on this rank
        img = rng.integers(0, 256, size=(IMG_HW[0], IMG_HW[1], 3), dtype=np.uint8)
        inp = prepare_inputs(proc, images=[img], prompts=f"request {i}", device=dev, stream=eng.stream)
        prompts[i] = inp["input_ids"].reshape(-1).tolist()
        kws[i] = {"pixel_values": inp["pixel_values"], "image_grid_thw": inp["image_grid_thw"]}
    for i in range(n_req):
        if prompts[i] is None:
            prompts[i] = [0]
    T = N_TEXT + 144
    dec_ms_box = []

    def make():
        g = BatchGenerator(model, proc, max_tokens=n_out, completion_batch_size=rows, prefill_batch_size=rows,
                           decode_slice=32)
        return g

    def run():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        toks = generate_sharded(make, prompts, n_out, kws)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, toks

    run()                      # warm-up (GEMM configurations are measured on first use, graphs captured)
    dt = 0.0
    for _ in range(args.steps):
        t, toks = run()
        dt += t / args.steps
    assert all(len(toks[i]) == n_out for i in shard_requests(n_req, world, rank))
    if args.dump_outputs:
        dump_output(args.dump_outputs, "c5_tokens", toks)      # every request's tokens (gathered over ranks)
    # device time of one lock-step step, from a dedicated slice of 64 steps on the warm engine
    step_ms = eng.last_decode_ms()
    t = torch.tensor([dt, step_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt, step_ms = t.tolist()
    peak, peak_src = _peaks()
    mean_ctx = T + n_out / 2
    bytes_step = W_BYTES_7B + rows * KV_BYTES_PER_POS_7B * mean_ctx
    out = {"workload": f"C5: Qwen2-VL-7B bf16, {n_req} concurrent requests ({rows} per GPU) over {world} GPU(s), "
                       f"1x336x336 image + 128 text tokens in, {n_out} out each, continuous batching "
                       "(lock-step rows, one weight stream per step), router: request i -> rank i mod N, "
                       f"seconds = mean of {args.steps} runs",
           "requests": n_req, "rows_per_gpu": rows, "seconds": dt,
           "requests_per_s": n_req / dt, "tokens_per_s": n_req * n_out / dt,
           "tokens_per_s_per_gpu": rows * n_out / dt,
           "decode_ms_per_step": step_ms,
           "roofline": {"kernel": "one lock-step decode step (28 x 7 kernels + head + sampler), all rows",
                        "bound": "hbm", "achieved": bytes_step / (step_ms / 1e3) / 1e9 if step_ms > 0 else None,
                        "peak": peak, "unit": "GB/s", "peak_source": peak_src,
                        "frac": (bytes_step / (step_ms / 1e3) / 1e9 / peak) if step_ms > 0 else None,
                        "algorithmic_bytes_per_step": bytes_step}}
    if bc:
        out["weight_broadcast"] = bc
    del model
    torch.cuda.empty_cache()
    return out


def c3_leg(dev, args):
    """BASELINE config 3: LLaVA-1.5-7B (CLIP-ViT-L/14-336 + Llama-7B geometry) bf16, batch = 8 images,
    prefill only: pinned-host pixel_values -> CLIP tower (23 of 24 blocks: feature layer -2) -> projector
    -> merge -> LM prefill of the 8 requests (576 image + 32 text tokens each) incl. the first token.
    The tower is fp32-accurate like the reference's (split-operand tcgen05 GEMMs: every Linear runs as
    W.x_hi + W.x_lo, i.e. 2x the algorithmic MMA flops; attention / LayerNorm in fp32 on the CUDA cores)."""
    import numpy as np
    import torch
    from mlx_vlm_b200.models.cache import make_prompt_cache
    from mlx_vlm_b200.models.llava import Model
    from mlx_vlm_b200.models.llava.config import llava_15_7b_config
    cfg = llava_15_7b_config()
    model = Model(cfg, device=dev).init_random(2)
    eng, lm = model.engine, model.language_model
    v, t = cfg.vision_config, cfg.text_config
    B, n_text = 8, 32
    P = (v.image_size // v.patch_size) ** 2
    rng = np.random.default_rng(11)
    pv_host = torch.from_numpy(rng.standard_normal((B, 3, v.image_size, v.image_size)).astype(np.float32)).pin_memory()
    text = rng.integers(3, 31000, size=n_text)
    ids = np.concatenate([text[:n_text // 2], np.full(P, cfg.image_token_index), text[n_text // 2:]])[None]
    T = ids.shape[1]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]

    def step():
        with torch.cuda.stream(eng.stream):
            pv = pv_host.to(dev, non_blocking=True)
        ev[0].record(eng.stream)
        feats = model.encode_image(pv)
        ev[1].record(eng.stream)
        embs = [model.get_input_embeddings(ids, pv, cached_image_features=feats[b:b + 1]).inputs_embeds for b in range(B)]
        if args.c3_sequential:      # A/B: one prefill call per request
            out = [lm(ids, inputs_embeds=embs[b], cache=make_prompt_cache(lm), logits_to_keep=1,
                      reserve_tokens=T + 8).logits for b in range(B)]
        else:                       # the 8 prompts in ONE pass over the weights (reference PromptProcessingBatch)
            rows, _ = lm.make_batch_cache(B, T + 8)
            out = lm.prefill_rows([ids] * B, embs, [lm.make_cache_row(rows.pool, b) for b in range(B)],
                                  reserve_tokens=T + 8)
        ev[2].record(eng.stream)
        eng.stream.synchronize()
        return ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), feats, out

    for _ in range(3):
        step()
    K = args.steps
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index or 0)     # this leg is the power-hungry one (dense tcgen05 work for ~0.1 s per step)
    sampler.start()
    t0 = time.perf_counter()
    tw, pf, per_step = 0.0, 0.0, []
    for _ in range(K):
        feats = out = None              # the previous step's outputs are freed before the next step allocates
        a, b, feats, out = step()
        tw += a
        pf += b
        per_step.append(round(b, 2))
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / K
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_output(args.dump_outputs, "c3_image_features", feats)
        if args.c3_sequential:
            dump_output(args.dump_outputs, "c3_prefill_logits", torch.cat(out))
        else:
            dump_output(args.dump_outputs, "c3_first_tokens", out)
    tw, pf = tw / K, pf / K
    E, I, nh = v.hidden_size, v.intermediate_size, v.num_attention_heads
    L = P + 1
    n_blocks = v.num_hidden_layers + 1 + cfg.vision_feature_layer if cfg.vision_feature_layer < 0 else cfg.vision_feature_layer
    H, Il = t.hidden_size, t.intermediate_size
    hd = H // t.num_attention_heads
    qkv = (t.num_attention_heads + 2 * t.num_key_value_heads) * hd
    tower_gf = (n_blocks * (2 * B * L * (4 * E * E + 2 * E * I) + 4 * B * L * L * E)
                + 2 * B * P * (3 * v.patch_size ** 2) * E + 2 * B * P * (E * H + H * H)) / 1e9
    lm_gf = B * (t.num_hidden_layers * (2 * T * (H * qkv + H * H + 3 * H * Il) + 2 * T * T * H) + 2 * t.vocab_size * H) / 1e9
    tpeak, tsrc = _tensor_peak()
    out = {"workload": f"C3: LLaVA-1.5-7B bf16 (random init), batch {B} x 336x336 images, prefill only: CLIP-L/14 tower "
                       f"({n_blocks} blocks, fp32-accurate split-operand GEMMs) + projector + merge + Llama-7B prefill "
                       f"of {B} requests x T={T} ({P} image + {n_text} text tokens), "
                       + ("one prefill call per request" if args.c3_sequential else "all requests in one batched prefill pass"),
           "tower_projector_ms": tw, "lm_prefill_ms": pf, "ms_per_step": tw + pf, "wall_ms_per_step": wall * 1e3,
           "lm_prefill_ms_per_step": per_step, "clocks": clocks,
           "prefill_img_tokens_per_sec": B * P / ((tw + pf) / 1e3),
           "tower_img_tokens_per_sec": B * P / (tw / 1e3),
           "h2d_bytes_per_step": int(pv_host.numel() * 4),
           "roofline": {"bound": "tensor", "unit": "TFLOP/s", "peak": tpeak, "peak_source": tsrc,
                        "tower": {"algorithmic_gflop": tower_gf, "achieved": tower_gf / tw, "frac": tower_gf / tw / tpeak,
                                  "executed_mma_gflop": "2x the Linear share (hi + lo operand halves)"},
                        "lm_prefill": {"algorithmic_gflop": lm_gf, "achieved": lm_gf / pf, "frac": lm_gf / pf / tpeak},
                        "achieved": (tower_gf + lm_gf) / (tw + pf), "frac": (tower_gf + lm_gf) / (tw + pf) / tpeak}}
    del model
    torch.cuda.empty_cache()
    return out


def c4_leg(dev, args):
    """BASELINE config 4: Idefics2-8B (SigLIP-SO400M + perceiver + Mistral-7B geometry) bf16, one request with
    4 images of 448x448 (4 x 1024 patches -> 4 x 64 latents = 256 image tokens) interleaved with 256 text
    tokens (T = 512), 256 greedy tokens out."""
    import numpy as np
    import torch
    from mlx_vlm_b200.models.cache import make_prompt_cache
    from mlx_vlm_b200.models.idefics2 import Model
    from mlx_vlm_b200.models.idefics2.config import idefics2_8b_config
    cfg = idefics2_8b_config()
    model = Model(cfg, device=dev).init_random(3)
    model.config.eos_token_id = []
    eng, lm = model.engine, model.language_model
    v, t, pc = cfg.vision_config, cfg.text_config, cfg.perceiver_config
    n_img, side, n_text, n_out = 4, 448, 256, 256
    nl = pc.resampler_n_latents
    rng = np.random.default_rng(13)
    pv_host = rng.standard_normal((1, n_img, 3, side, side)).astype(np.float32)
    text = rng.integers(3, 31000, size=n_text)
    seg = n_text // (n_img + 1)
    parts = []
    for i in range(n_img):   # text / image / text / image ... (interleaved, like the processor's <image> expansion)
        parts += [text[i * seg:(i + 1) * seg], np.full(nl, cfg.image_token_index)]
    parts.append(text[n_img * seg:])
    ids = np.concatenate(parts)[None]
    T = ids.shape[1]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

    def step():
        ev[0].record(eng.stream)
        feats = model.encode_image(pv_host)          # host pixels: pinned H2D inside
        ev[1].record(eng.stream)
        emb = model.get_input_embeddings(ids, pv_host, cached_image_features=feats)
        cache = make_prompt_cache(lm)
        out = lm(ids, inputs_embeds=emb.inputs_embeds, cache=cache, logits_to_keep=1, reserve_tokens=T + n_out + 1)
        ev[2].record(eng.stream)
        lm.fused_greedy_decode_n(n_out, cache, reserve_tokens=T + n_out + 1)
        ev[3].record(eng.stream)
        eng.stream.synchronize()
        return (ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3])), feats, out.logits

    for _ in range(2):
        step()
    K = args.steps
    l0 = eng.launch_count
    acc = [0.0, 0.0, 0.0]
    for _ in range(K):
        feats = logits = None           # the previous step's outputs are freed before the next step allocates
        times, feats, logits = step()
        for i, x in enumerate(times):
            acc[i] += x / K
    launches = (eng.launch_count - l0) / K
    if args.dump_outputs:
        dump_output(args.dump_outputs, "c4_image_features", feats)
        dump_output(args.dump_outputs, "c4_prefill_logits", logits)
        dump_output(args.dump_outputs, "c4_tokens", _token_log(eng, n_out + 1))
    tw, pf, dec = acc
    H, Il = t.hidden_size, t.intermediate_size
    hd = H // t.num_attention_heads
    qkv = (t.num_attention_heads + 2 * t.num_key_value_heads) * hd
    w_bytes = 2 * (t.num_hidden_layers * (H * qkv + H * H + 3 * H * Il) + t.vocab_size * H)
    kv_pos = 2 * t.num_key_value_heads * hd * 2 * t.num_hidden_layers
    bytes_step = w_bytes + kv_pos * (T + n_out / 2)
    step_ms = dec / n_out
    peak, psrc = _peaks()
    out = {"workload": f"C4: Idefics2-8B bf16 (random init), 1 request, {n_img} x {side}x{side} images ({n_img} x "
                       f"{(side // v.patch_size) ** 2} patches -> {n_img * nl} image tokens) interleaved with {n_text} text "
                       f"tokens (T={T}), {n_out} greedy tokens out",
           "tower_connector_ms": tw, "merge_prefill_ms": pf, "decode_ms": dec, "decode_ms_per_token": step_ms,
           "decode_tokens_per_sec": n_out / (dec / 1e3), "prefill_img_tokens_per_sec": n_img * nl / ((tw + pf) / 1e3),
           "gpu_launches_per_request": launches,
           "roofline": {"kernel": "decode step of the Mistral-7B geometry (32 q / 8 kv heads)", "bound": "hbm",
                        "achieved": bytes_step / (step_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s", "peak_source": psrc,
                        "frac": bytes_step / (step_ms / 1e3) / 1e9 / peak, "algorithmic_bytes_per_step": bytes_step}}
    del model
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="skip the C5 leg (Qwen2-VL-7B continuous batching)")
    ap.add_argument("--no-c3", action="store_true", help="skip the C3 leg (LLaVA-1.5-7B, 8 images, prefill only)")
    ap.add_argument("--c3-sequential", action="store_true", help="C3: prefill the 8 requests one by one (A/B)")
    ap.add_argument("--no-c4", action="store_true", help="skip the C4 leg (Idefics2-8B, 4 images, 256 out)")
    ap.add_argument("--c5-rows", type=int, default=8, help="concurrent requests per GPU in the C5 leg")
    ap.add_argument("--c5-out", type=int, default=512)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-pdl", action="store_true")
    ap.add_argument("--pdl", action="store_true")
    ap.add_argument("--no-mega", action="store_true")
    ap.add_argument("--mega-mode", type=int, default=None,
                    help="decode kernel: 0 per-phase kernels, 1 k_mega (CUDA cores), 2 k_mega_tc (tcgen05)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what each leg's last timed step returned as DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the outputs of the b200 implementation")

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        args.dump_outputs = None          # rank 0 writes the outputs (C5 tokens are gathered from every rank)
    elif args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    import numpy as np
    import torch

    config = {"workload": "C2: Qwen2-VL-2B bf16, 1x336x336 image (144 img tokens) + 128 text "
                          "tokens in (T=272), 512 greedy tokens out, batch 1",
              "global_batch": world, "parallelism": f"dp{world} (one replica per GPU, "
              "no per-step collective)", "l2": "weights streamed per token (3.09 GB) exceed the "
              "126 MB L2; no flush needed"}

    # ------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import qwen2vl as O
        c = O.qwen2_vl_2b()
        W = O.init_weights(c, 0)
        n_dec = 4
        vals = []
        for i in range(args.warmup + args.steps):
            r = cpu_reference_run(W, n_dec)
            if i >= args.warmup:
                vals.append(r)
        dec_s = sum(v["decode_s"] for v in vals)
        tps = len(vals) * n_dec / dec_s
        line = {"impl": "reference", "metric": "decode_tokens_per_sec", "value": tps,
                "unit": "tokens/s", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup,
                "ms_per_step": 1e3 * sum(v["decode_s"] + v["prefill_s"] for v in vals) / len(vals),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic", "config": config,
                "prefill_img_tokens_per_sec": len(vals) * 144 / sum(v["prefill_s"] for v in vals),
                "cpu_baseline": {"value": tps, "unit": "tokens/s", "cores": vals[0]["cores"],
                                 "kind": "port", "cpu": _cpu_model(),
                                 "sample": f"per step: C2 prompt ViT+prefill once, {n_dec} decode "
                                           "steps (oracle = CPU restatement of the reference's "
                                           "MLX-CPU path; mlx is not installable offline)"},
                "e2e": {"value": tps, "unit": "tokens/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------ B200 arm
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from mlx_vlm_b200 import generate as api_generate
    from mlx_vlm_b200.models.cache import make_prompt_cache
    from mlx_vlm_b200.utils import load_synthetic, prepare_inputs

    model, processor = load_synthetic("qwen2-vl-2b", seed=0, device=dev, n_text_tokens=N_TEXT)
    model.config.eos_token_id = []  # benchmark: EOS ignored (fixed 512 tokens out)
    eng = model.engine
    if args.no_graph:
        eng.set_graph(False)
    if args.no_pdl:
        eng.set_pdl(False)
    if args.pdl:
        eng.set_pdl(True)
    if args.no_mega:
        eng.set_mega(False)
    if args.mega_mode is not None:
        eng.set_mega(args.mega_mode)
    bcast = None
    if world > 1:
        # the single collective of the design: rank 0's packed weight arena, ONE NCCL broadcast
        from mlx_vlm_b200.parallel import broadcast_packed
        torch.cuda.synchronize()
        dist.barrier()
        tb = time.perf_counter()
        nb = broadcast_packed(model.packed_weights, src=0)
        torch.cuda.synchronize()
        dtb = time.perf_counter() - tb
        bcast = {"bytes": nb, "seconds": dtb, "GB_per_s": nb / dtb / 1e9, "calls": 1}

    rng = np.random.default_rng(0)
    image = rng.integers(0, 256, size=(IMG_HW[0], IMG_HW[1], 3), dtype=np.uint8)
    prompt = "Describe this image in detail."
    inputs = prepare_inputs(processor, images=[image], prompts=prompt, device=dev, stream=eng.stream)
    ids = inputs["input_ids"]
    pvd = inputs["pixel_values"]
    grid = inputs["image_grid_thw"]
    eng.stream.synchronize()
    T = int(ids.shape[1])
    assert T == N_TEXT + 144, T

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

    def device_step():
        """one request with inputs resident in HBM; returns (prefill_ms, decode_ms, embeddings, prefill logits)."""
        cache = make_prompt_cache(model.language_model)
        ev[0].record(eng.stream)
        emb = model.get_input_embeddings(ids, pvd, image_grid_thw=grid)
        out = model.language_model(ids, inputs_embeds=emb.inputs_embeds, cache=cache,
                                   position_ids=emb.position_ids, rope_deltas=emb.rope_deltas,
                                   logits_to_keep=1, reserve_tokens=T + N_OUT + 1)
        ev[1].record(eng.stream)
        model.language_model.fused_greedy_decode_n(N_OUT, cache, reserve_tokens=T + N_OUT + 1)
        ev[2].record(eng.stream)
        eng.stream.synchronize()
        return ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), emb.inputs_embeds, out.logits

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        device_step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = eng.launch_count
    t0 = time.perf_counter()
    pre_ms, dec_ms = 0.0, 0.0
    for _ in range(args.steps):
        embeds = logits = None          # the previous step's outputs are freed before the next step allocates
        a, b, embeds, logits = device_step()
        pre_ms += a
        dec_ms += b
    barrier()
    wall = time.perf_counter() - t0
    launches = eng.launch_count - l0
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_output(args.dump_outputs, "c2_inputs_embeds", embeds)
        dump_output(args.dump_outputs, "c2_prefill_logits", logits)
        dump_output(args.dump_outputs, "c2_tokens", _token_log(eng, N_OUT + 1))
        dump_output(args.dump_outputs, "c2_last_logprobs", eng.snapshot("logprobs"))

    # ---- e2e through the public API with a host image --------------------------
    def e2e_step():
        t = time.perf_counter()
        r = api_generate(model, processor, prompt, image=[image], max_tokens=N_OUT)
        torch.cuda.synchronize()
        return time.perf_counter() - t, r

    for _ in range(min(args.warmup, 2)):
        e2e_step()
    barrier()
    e2e_t, e2e_gen_tps, e2e_prompt_tps = 0.0, [], []
    for _ in range(args.steps):
        dt, r = e2e_step()
        e2e_t += dt
        e2e_gen_tps.append(r.generation_tps)
        e2e_prompt_tps.append(r.prompt_tps)
        assert r.generation_tokens == N_OUT
    barrier()
    if args.dump_outputs:
        dump_output(args.dump_outputs, "e2e_last_logprobs", r.logprobs)

    c5 = None
    if not args.no_c5:
        rows2b = lockstep_2b(world, rank, dev, args, model, processor, ids, pvd, grid)
        c5 = c5_leg(world, rank, dev, args)
        c5["qwen2_vl_2b_rows"] = rows2b

    c3 = c3_leg(dev, args) if (rank == 0 and not args.no_c3) else None
    c4 = c4_leg(dev, args) if (rank == 0 and not args.no_c4) else None
    if world > 1:
        dist.barrier()

    stats = torch.tensor([dec_ms, pre_ms, wall, e2e_t], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    dec_ms, pre_ms, wall, e2e_t = stats.tolist()

    if rank == 0:
        K = args.steps
        dec_tps = world * K * N_OUT / (dec_ms / 1e3)
        img_tps = world * K * 144 / (pre_ms / 1e3)
        peak, peak_src = _peaks()
        tpeak, tpeak_src = _tensor_peak()
        traffic, traffic_src = _ncu_traffic()
        pre_tflops = (VIT_GFLOP + PREFILL_GFLOP_T272) / (pre_ms / K)   # GFLOP / ms = TFLOP/s
        mean_ctx = T + N_OUT / 2
        bytes_per_step = W_BYTES_2B + KV_BYTES_PER_POS * mean_ctx
        step_ms = dec_ms / (K * N_OUT)
        achieved = bytes_per_step / (step_ms / 1e3) / 1e9
        line = {
            "metric": "decode_tokens_per_sec", "value": dec_tps, "unit": "tokens/s",
            "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": (pre_ms + dec_ms) / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config,
            "prefill_img_tokens_per_sec": img_tps,
            "prefill_ms": pre_ms / K, "decode_ms_per_token": step_ms,
            "wall_s_timed_region": wall,
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": world * K * N_OUT / e2e_t, "unit": "tokens/s",
                    "definition": "512 generated tokens / wall time of generate(model, processor, "
                                  "prompt, image=[HxWx3 uint8 host array]) incl. host "
                                  "preprocessing, H2D, ViT, prefill, decode, per-token D2H",
                    "generation_tps_api": statistics.mean(e2e_gen_tps),
                    "prompt_tps_api": statistics.mean(e2e_prompt_tps),
                    "h2d_bytes_per_step": int(576 * 1176 * 4 + T * 4 + 3 * T * 4),
                    "d2h_bytes_per_step": int(N_OUT * 4)},
            "roofline": {"kernel": "k_mega (persistent decode-step kernel: 28 x {qkv, attention, "
                                   "o_proj, gate/up, down} + head + sampler), one launch = one "
                                   "token",
                         "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": bytes_per_step,
                         "traffic": traffic, "traffic_source": traffic_src},
            # the other half of the metric: ViT + merge + LM prefill (T=272) on the tensor cores
            "roofline_prefill": {"kernels": "ViT (32 blocks) + merge + LM prefill (28 layers, T=272): "
                                            "tcgen05 GEMMs + tcgen05 attention + row ops",
                                 "bound": "tensor", "achieved": pre_tflops, "peak": tpeak,
                                 "unit": "TFLOP/s", "frac": pre_tflops / tpeak, "peak_source": tpeak_src,
                                 "algorithmic_gflop": VIT_GFLOP + PREFILL_GFLOP_T272},
            "parity": {"per_op": "rel-L2 <= 1e-3 vs oracle on identical inputs (tests/test_kernels_gpu.py)",
                       "integer": "bit-exact (merge indices, rope ids, cache offsets)",
                       "e2e": "deep bf16 chain: |cuda-oracle| <= 1.5 x |oracle_bf16 - exact fp32| "
                              "(tests/_util.cmp_noise; C2 as benched: tests/test_gate_gpu.py)",
                       "oracle": "CPU restatement pinned on the reference's own source + HF fp32; "
                                 "mlx rounding points unpinned (mlx not installable offline)"},
        }
        if bcast is not None:
            line["weight_broadcast"] = bcast
        if c5 is not None:
            line["c5"] = c5
        if c3 is not None:
            line["c3"] = c3
        if c4 is not None:
            line["c4"] = c4
        if not args.no_cpu_baseline and world == 1:
            W = _engine_weights_to_oracle(model, __import__("oracle.qwen2vl", fromlist=["x"]).qwen2_vl_2b())
            r = cpu_reference_run(W, 6)
            line["cpu_baseline"] = {
                "value": r["decode_tps"], "unit": "tokens/s", "cores": r["cores"], "kind": "port",
                "cpu": _cpu_model(),
                "prefill_img_tokens_per_sec": r["img_tps"],
                "sample": "same weights/prompt as the GPU run: ViT+merge+prefill (T=272) once, "
                          "6 decode steps, torch-CPU fp32 matmuls with bf16 rounding points "
                          "(oracle port of the reference's MLX-CPU path)"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
