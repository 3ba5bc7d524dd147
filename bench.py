#!/usr/bin/env python
"""bench.py — preference-pairs/sec of one full LLaVA-1.5-7B DPO optimisation step on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]            (N=1)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = policy forward on chosen+rejected (CLIP -> projector -> splice -> 32 decoder layers ->
lm_head -> log-prob gather), DPO loss + gradient, full backward, ZeRO-2 gradient reduction and the
fused fp32 AdamW, on BASELINE.json configs[1]: 8 synthetic pairs per GPU, 336x336 images,
48-token prompt + 512-token responses (T = 1135), bf16, random-init weights at true dimensions.

`value`  : whole-job pairs/s with the step's inputs already resident in HBM.
`e2e`    : same metric through the public call DPOStepEngine.train_step() with HOST (pinned) buffers:
           H2D of ids/labels/images/ref-logps and a D2H read of the loss inside the timed region.
`roofline`: dominant kernel = the tcgen05 GEMM; achieved = sum(2MNK) / sum(CUDA-event durations) of
           every GEMM launch of one instrumented step, against MEASURED_PEAKS.json.
`cpu_baseline` / `--impl reference`: the UNMODIFIED reference staged under oracle/_ref (oracle/stage_ref.py; the
           oracle port only if that staging is absent) on the host cores, on a bounded sample: full-width config-(a)
           steps at 2 and 8 decoder layers after a warm-up, min of 3, extrapolated to 32 layers, raw timings in the
           line (see cpu_reference_pairs_per_sec); thread count calibrated against the container's real CPU quota.
`parity_full_width`: checker leg — the CUDA path vs the oracle on the same full-width 1-layer model (log-probs,
           loss, gradients), with the reference's own bf16-vs-fp32 gap beside it.
Side workloads (not the headline line): `--lora` (BASELINE config e), `--omnilmm` (config d downstream of the
vision tower).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

PAIRS_PER_GPU = 8
PROMPT_LEN, RESP_LEN, IMAGE_POS = 48, 512, 35


def flops_per_pair(T):
    """BASELINE.md §3: F_pair = 3*2*F_seq(T) + F_clip + 3*F_proj (algorithmic, no recompute)."""
    n_dec = 32 * (4 * 4096 ** 2 + 3 * 4096 * 11008)
    n_head = 4096 * 32000
    f_seq = 2 * (n_dec + n_head) * T + 32 * 4 * T * T * 4096 * 0.5
    f_clip = 2 * 23 * (4 * 1024 ** 2 + 2 * 1024 * 4096) * 577 + 23 * 4 * 577 ** 2 * 1024 + 2 * 588 * 1024 * 576
    f_proj = 2 * (1024 * 4096 + 4096 ** 2) * 576
    return 3 * 2 * f_seq + f_clip + 3 * f_proj


def measured_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("bf16_tflops_sustained", 1400.0), d.get("bf16_tflops", 1590.0), "measured"
    return 1400.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def synthetic_batch(rank, step, B):
    """SURVEY.md §8d canonical inputs (seed 1234 + 1000*rank + step), host tensors (pinned)."""
    g = torch.Generator().manual_seed(1234 + 1000 * rank + step)
    L = PROMPT_LEN + RESP_LEN
    ids = torch.empty((2 * B, L), dtype=torch.int64)
    labels = torch.full((2 * B, L), -100, dtype=torch.int64)
    for i in range(B):
        prompt = torch.randint(3, 32000, (PROMPT_LEN,), generator=g)
        prompt[0] = 1
        prompt[IMAGE_POS] = -200
        for row in (i, B + i):
            resp = torch.randint(3, 32000, (RESP_LEN,), generator=g)
            resp[-1] = 2
            ids[row] = torch.cat([prompt, resp])
            labels[row, PROMPT_LEN:] = resp
    images = torch.randn(B, 3, 336, 336, generator=g)
    return {"concatenated_input_ids": ids.pin_memory(), "concatenated_labels": labels.pin_memory(),
            "images": images.pin_memory(), "beta": 0.1}


def synthetic_omni_batch(rank, step, B, dims, n_vision_tokens=1024):
    """Config (d) shape downstream of the vision tower: the same 48-token prompt / 512-token responses, the image slot
    expanded in place to <im_start> <im_patch>*64 <im_end> (omnilmm token layout), and the tower's output tokens
    [B, 1024, 1792] (448 px / 14) as `images`."""
    g = torch.Generator().manual_seed(1234 + 1000 * rank + step)
    Q = dims.num_query
    P = PROMPT_LEN - 1 + Q + 2
    L = P + RESP_LEN
    ids = torch.empty((2 * B, L), dtype=torch.int64)
    labels = torch.full((2 * B, L), -100, dtype=torch.int64)
    for i in range(B):
        text = torch.randint(3, 32000, (PROMPT_LEN,), generator=g)
        text[0] = 1
        slot = torch.cat([torch.tensor([dims.im_start_token]), torch.full((Q,), dims.im_patch_token),
                          torch.tensor([dims.im_end_token])])
        prompt = torch.cat([text[:IMAGE_POS], slot, text[IMAGE_POS + 1:]])
        for row in (i, B + i):
            resp = torch.randint(3, 32000, (RESP_LEN,), generator=g)
            resp[-1] = 2
            ids[row] = torch.cat([prompt, resp])
            labels[row, P:] = resp
    tokens = torch.randn(B, n_vision_tokens, dims.vision_width, generator=g).to(torch.bfloat16)
    return {"concatenated_input_ids": ids.pin_memory(), "concatenated_labels": labels.pin_memory(),
            "images": tokens.pin_memory(), "beta": 0.1}


def omni_flops_per_pair(d, T, n_vision_tokens=1024):
    """Algorithmic FLOPs of one pair downstream of the tower: 3 x (2 sequences through the GQA decoder + head) +
    3 x resampler (one image per pair)."""
    H, F, KV, V = d.hidden_size, d.intermediate_size, d.kv_size, d.vocab_size
    n_dec = d.num_layers * (2 * H * H + 2 * H * KV + 3 * H * F)
    f_seq = 2 * (n_dec + H * V) * T + d.num_layers * 4 * T * T * H * 0.5
    N, Q = n_vision_tokens, d.num_query
    f_res = 2 * N * d.vision_width * H + 2 * 2 * N * H * H + 2 * Q * H * H + 4 * Q * N * H + 2 * 2 * Q * H * H
    return 3 * 2 * f_seq + 3 * f_res


# ------------------------------------------------------------------------------------------------
# CPU arm: oracle port of the reference path on the host cores, bounded sample
# ------------------------------------------------------------------------------------------------
CHECKER_PARAM_SCALE = 0.3   # std multiplier of oracle.make_params for the full-width checker model: random matrices at
                            # the stock scale give per-token log-probs of -15 and attention scores of std ~10 at
                            # h=4096 — an ill-conditioned network on which two valid evaluation orders (fp32 vs the
                            # reference's own bf16 op order) already differ by 1e-2 in summed log-prob; at 0.3 the
                            # logits look like a real checkpoint's (mean per-token logp -10.9 ~ ln 32000) and the two
                            # orders agree to 5e-5 (tools/cpu_fullwidth_inherent.py)


def full_width_case(num_layers, dtype=torch.float32, cfg=None):
    """The oracle-side model / batch of the cpu_baseline leg: full width (or `cfg`'s dims), config (a) shape (1 pair,
    R=64, T=687)."""
    import dataclasses
    from oracle import llava_dpo_oracle as O
    cfg = O.OracleConfig(num_layers=num_layers) if cfg is None else dataclasses.replace(cfg, num_layers=num_layers)
    p = O.make_params(cfg, seed=0, dtype=dtype, scale=CHECKER_PARAM_SCALE)
    for k in p:
        if k.startswith(O.TRAINABLE_PREFIXES):
            p[k].requires_grad_(True)
    batch = O.synthetic_pair_batch(cfg, 1, 48, 64, seed=1234, image_pos=35)
    batch["images"] = batch["images"].to(dtype)
    batch["ref_win_logp"] = torch.tensor([-700.0])
    batch["ref_rej_logp"] = torch.tensor([-690.5])
    return cfg, p, batch


def gpu_full_width_parity(p, cfg, batch, out):
    """Checker leg: the CUDA path on the SAME full-width 1-layer model / batch the oracle port just ran
    (h=4096, ffn=11008, vocab=32000, CLIP-L 23 layers; config (a) shape) — log-probs, loss and gradients; plus the
    oracle in the reference's bf16 op order as the yardstick of what bf16 storage costs by itself."""
    from oracle import llava_dpo_oracle as O
    from rlaifv_b200 import ops
    from rlaifv_b200.model import LlavaDims, LlavaDPOPolicy
    pol = LlavaDPOPolicy(LlavaDims(num_layers=cfg.num_layers), "cuda", hf_state={k: v.detach() for k, v in p.items()})
    o = pol.forward_logps(batch["concatenated_input_ids"], batch["concatenated_labels"], batch["images"].float(),
                          keep_stash=True)
    B = batch["images"].shape[0]
    lp = o["logp"]
    losses, _, _, dpw, dpr, out9 = ops.dpo_loss(lp[:B].contiguous(), lp[B:].contiguous(), batch["ref_win_logp"].cuda(),
                                                batch["ref_rej_logp"].cuda(), 0.1)
    pol.backward_logps(torch.cat([dpw, dpr]).contiguous())
    pol.finalize_embed_grad()
    torch.cuda.synchronize()
    with torch.no_grad():
        pb = {k: v.detach().to(torch.bfloat16) for k, v in p.items()}
        ob = O.policy_logps(pb, cfg, batch["concatenated_input_ids"], batch["concatenated_labels"],
                            batch["images"].to(torch.bfloat16))
    ref_lp = out["logp"].detach().double()
    mask = (out["labels"][:, 1:] != -100)
    pt_ref = out["per_token_logps"].detach().double()[mask]
    pt_gpu = o["per_token_logps"].double().cpu()[mask]
    pt_bf = ob["per_token_logps"].double()[mask]
    relmax = lambda a, b: float(((a - b).abs() / b.abs()).max())
    grads = pol.store.hf_grad_views()
    gerr = {}
    for name in ("model.mm_projector.0.weight", "model.mm_projector.2.weight", "model.layers.0.self_attn.q_proj.weight",
                 "model.layers.0.self_attn.o_proj.weight", "model.layers.0.mlp.gate_proj.weight",
                 "model.layers.0.mlp.down_proj.weight", "model.layers.0.input_layernorm.weight", "model.norm.weight",
                 "lm_head.weight"):
        ref = p[name].grad.detach().double()
        got = grads[name].double().cpu().view_as(ref)
        gerr[name] = float((got - ref).norm() / (ref.norm() + 1e-300))
    res = {"shape": "1 decoder layer at full width, 1 pair, R=64 (T=687); oracle.make_params scale %g" % CHECKER_PARAM_SCALE,
           "logp_oracle_fp32": ref_lp.tolist(), "logp_gpu": lp.double().cpu().tolist(),
           "logp_oracle_bf16_order": ob["logp"].double().tolist(),
           "logp_rel_err": relmax(lp.double().cpu(), ref_lp),
           "logp_rel_err_inherent_bf16_order": relmax(ob["logp"].double(), ref_lp),
           "per_token_logp_max_abs_err": float((pt_gpu - pt_ref).abs().max()),
           "per_token_logp_max_abs_err_inherent_bf16_order": float((pt_bf - pt_ref).abs().max()),
           "loss_oracle": float(out["loss"].detach()), "loss_gpu": float(out9[0]),
           "grad_rel_l2_err": gerr}
    del pol
    torch.cuda.empty_cache()
    return res


def usable_cores():
    """Host cores this process may really use: min(cpu_count, scheduler affinity, cgroup cpu quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(math.ceil(int(quota) / int(period)))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def pick_cpu_threads():
    """Thread count that gives the reference's CPU path its best throughput on this box: a 2048^3 fp32 matmul is
    timed at a few candidate counts (a container can report 128 CPUs and still be scheduled on far fewer, where 128
    threads thrash)."""
    n = usable_cores()
    cands = sorted({c for c in (n, n // 2, 64, 32, 16, 8, 4) if 1 <= c <= n}, reverse=True)
    a = torch.randn(2048, 2048)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        a @ a
        t0 = time.perf_counter()
        for _ in range(3):
            a @ a
        t = time.perf_counter() - t0
        if t < best_t * 0.95:           # prefer more threads unless fewer are clearly faster
            best, best_t = c, t
    torch.set_num_threads(best)
    return best


REF_ARM_LAYERS = (2, 8)     # full-width decoder depths that are timed; the 32-layer step is extrapolated linearly
                            # (a 6-layer lever arm: with (2, 4) the x14 extrapolation turned 3 % timing noise into 15 %)


def _time_cpu_steps(step_fn, warmup, reps):
    """`warmup` untimed passes (first-touch page faults of parameters / gradients / AdamW state / activations, oneDNN
    primitive creation), then `reps` timed ones; returns the list of wall-clock seconds."""
    for _ in range(warmup):
        step_fn()
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        step_fn()
        out.append(time.perf_counter() - t0)
    return out


def _reference_step_fn(nl, cfg=None):
    """One DPO optimisation step of the UNMODIFIED reference (staged under oracle/_ref by oracle/stage_ref.py) on
    torch-CPU fp32 at full width with `nl` decoder layers, config (a) shape: the reference's collator ->
    get_beta_and_logps(is_llava15=True) [prepare_inputs_labels_for_multimodal -> LlavaLlamaForCausalLM.forward ->
    get_batch_logps] -> dpo_loss -> backward -> torch.optim.AdamW.step (BASELINE.md §4)."""
    from oracle import llava_dpo_oracle as O       # input synthesis only (SURVEY §8d canonical inputs)
    from oracle import stage_ref
    import dataclasses
    R = stage_ref.import_reference()
    cfg = O.OracleConfig(num_layers=nl) if cfg is None else dataclasses.replace(cfg, num_layers=nl)
    model = stage_ref.build_reference_model(R, cfg, None)      # HF random init at true dimensions
    model.train()
    opt = torch.optim.AdamW([p for p in model.parameters() if p.requires_grad], lr=5e-7, weight_decay=0.01)
    batch = O.synthetic_pair_batch(cfg, 1, PROMPT_LEN, 64, seed=1234, image_pos=IMAGE_POS)

    class Tok:
        pad_token_id = 0

    class Args:
        dpo_use_average = False
        dpo_token_weighted = False
        task = "DPO"

    ids, labs = batch["concatenated_input_ids"], batch["concatenated_labels"]
    inst = []
    for kind, row in (("rej", 1), ("win", 0)):
        inst.append({"input_ids": ids[row].clone(), "labels": labs[row].clone(), "image": batch["images"][0],
                     f"ref_{kind}_logp": -700.0 if kind == "win" else -690.5, f"ref_{kind}_avg_logp": -10.9,
                     f"ref_{kind}_per_token_logp": [0.0] * (ids.shape[1] + 600)})
    data = R["DataCollatorForDPODataset"](tokenizer=Tok(), beta=0.1, mod_token_weight=1.0)([tuple(inst)])

    def step():
        opt.zero_grad(set_to_none=True)
        pw, pr, rw, rr, beta = R["get_beta_and_logps"](dict(data), model, Args(), is_llava15=True)
        losses, _, _ = R["dpo_loss"](pw, pr, rw, rr, beta=beta)
        loss = losses.mean()
        loss.backward()
        opt.step()
        return float(loss)
    return step


def _port_step_fn(nl, cfg=None):
    """Fallback when oracle/_ref is not staged: the oracle port of the same path (kind "port")."""
    from oracle import llava_dpo_oracle as O
    cfg, p, batch = full_width_case(nl, torch.float32, cfg=cfg)
    names = O.trainable_names(p)
    state = {k: [torch.zeros_like(p[k]), torch.zeros_like(p[k])] for k in names}

    def step():
        for k in names:
            p[k].grad = None
        out = O.dpo_step(p, cfg, batch, beta=0.1)
        out["loss"].backward()
        with torch.no_grad():
            for k in names:
                new_p, m, v = O.adamw_update(p[k], p[k].grad, state[k][0], state[k][1], 1, 5e-7)
                p[k].copy_(new_p)
                state[k][0], state[k][1] = m, v
        return float(out["loss"])
    return step


def cpu_reference_pairs_per_sec(reps=3, warmup=1):
    """The reference arm / cpu_baseline leg: full-width (h=4096, ffn=11008, vocab=32000, CLIP-L 23 layers, 336 px)
    config-(a) step (1 pair, 64-token responses, T=687), fp32, timed at 2 and 8 decoder layers after a warm-up pass
    each (min of `reps`), extrapolated linearly to the 32-layer model: t32 = t8 + 24 * (t8 - t2) / 6.
    Returns (pairs/s, threads, kind, sample description, raw timings)."""
    from oracle import stage_ref
    threads = pick_cpu_threads()
    kind = "reference" if stage_ref.available() else "port"
    make = _reference_step_fn if kind == "reference" else _port_step_fn
    raw, best = {}, {}
    for nl in REF_ARM_LAYERS:
        fn = make(nl)
        raw[nl] = _time_cpu_steps(fn, warmup, reps)
        best[nl] = min(raw[nl])
        del fn
        import gc
        gc.collect()
    lo, hi = REF_ARM_LAYERS
    t_layer = max((best[hi] - best[lo]) / (hi - lo), 1e-9)
    t_full = best[hi] + (32 - hi) * t_layer
    src = ("the unmodified reference staged under oracle/_ref (collator -> get_beta_and_logps -> dpo_loss -> backward "
           "-> torch.optim.AdamW)" if kind == "reference" else "oracle port of the reference path (oracle/_ref not staged)")
    sample = ("%s, torch-CPU float32, full width, config (a) shape: 1 pair, R=64 (T=687); %d warm-up + %d timed steps at "
              "%d and %d decoder layers (min %.2fs / %.2fs), extrapolated linearly to 32 layers (%.2fs per layer => "
              "%.1fs per step); %d torch threads (matmul calibration; os.cpu_count()=%s)"
              % (src, warmup, reps, lo, hi, best[lo], best[hi], t_layer, t_full, threads, os.cpu_count()))
    timings = {"layers_%d_s" % nl: [round(t, 3) for t in raw[nl]] for nl in REF_ARM_LAYERS}
    timings.update(per_layer_s=round(t_layer, 4), extrapolated_step_s=round(t_full, 2))
    return 1.0 / t_full, threads, kind, sample, timings


def run_reference_arm(args, rank):
    """`bench.py --impl reference`: rank 0 alone runs; other ranks exit 0 without work. A "step" of this arm is the
    bounded sample described in cpu_reference_pairs_per_sec; K and W are capped (3 / 1) so that the run ends within
    a few minutes whatever the driver passes."""
    if rank != 0:
        return
    reps, warm = max(1, min(args.steps, 3)), max(1, min(args.warmup, 1))
    value, cores, kind, sample, timings = cpu_reference_pairs_per_sec(reps=reps, warmup=warm)
    line = {"impl": "reference", "metric": "preference-pairs/sec LLaVA-1.5-7B DPO step", "value": value,
            "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "LLaVA-1.5-7B DPO step, reference CPU path (config (a) shape: 1 pair, 336px, 64-tok "
                                   "responses; full width, 2- and 8-layer steps extrapolated to 32 layers)",
                       "timed_steps_per_depth": reps, "warmup_steps_per_depth": warm, "same_config_as_b200_arm": False,
                       "note": "BASELINE.json configs[0] is the reference's CPU-runnable case; configs[1] (8 pairs, "
                               "512-tok) would take ~15 min per CPU step"},
            "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": kind, "sample": sample,
                             "timings": timings},
            "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def full_width_parity_report():
    """Checker leg (not timed): oracle fp32 fwd+bwd on the full-width 1-layer model, then the CUDA path on the same
    weights / batch."""
    from oracle import llava_dpo_oracle as O
    cfg, p, batch = full_width_case(1, torch.float32)
    out = O.dpo_step(p, cfg, batch, beta=0.1)
    out["loss"].backward()
    try:
        return gpu_full_width_parity(p, cfg, batch, out)
    except Exception as exc:                      # the checker must never take the bench line down
        return {"error": "%s: %s" % (type(exc).__name__, exc)}


# ------------------------------------------------------------------------------------------------
def eva_flops_per_image(e, batch_tokens=None):
    """Algorithmic forward FLOPs of the EVA tower for one 448 px image (63 live blocks, 1025 tokens)."""
    C, Hd, S = e.embed_dim, e.mlp_hidden, e.n_tokens + 1
    per_block = 2 * S * (4 * C * C + 2 * C * Hd) + 4 * S * S * C
    return e.live_blocks * per_block + 2 * e.n_tokens * e.patch_k * C


DUMP_SAMPLE = 1 << 21      # parameter / gradient entries --dump-outputs writes per store (8 MB per array in float32)


def dump_outputs(out_dir, metrics, policy):
    """`--dump-outputs DIR`: what the last timed step computed, as float32 .npy files — `metrics.npy`, the 9 values
    train_step returned (engine.METRIC_NAMES order), and `params.npy` / `grads.npy`, the bf16 parameters after that
    step's AdamW update and the gradients it produced, at DUMP_SAMPLE fixed, seeded positions of the flat store
    (`lora_params.npy` / `lora_grads.npy` likewise for the adapters of a LoRA run)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "metrics.npy"), metrics.float().cpu().numpy())
    stores = [("", policy.store)]
    if getattr(policy, "lora", None) is not None:
        stores.append(("lora_", policy.lora))
    for prefix, st in stores:
        n = st.flat.numel()
        g = torch.Generator().manual_seed(0)
        idx = torch.randint(0, n, (min(DUMP_SAMPLE, n),), generator=g).sort().values.to(st.flat.device)
        np.save(os.path.join(out_dir, prefix + "params.npy"), st.flat[idx].float().cpu().numpy())
        np.save(os.path.join(out_dir, prefix + "grads.npy"), st.grad[idx].float().cpu().numpy())


def run_workload(args, rank, local_rank, world, lora=False, omnilmm=False, steps=None, warmup=None, extras=False,
                 dump_dir=None):
    """One measured workload -> the JSON line (dict). `extras`: a run for one of the `extra` sub-records.
    `dump_dir`: where rank 0 writes the outputs of the last timed step (dump_outputs)."""
    from rlaifv_b200 import lib, ops
    from rlaifv_b200.engine import DPOStepEngine
    from rlaifv_b200.model import LlavaDims, LlavaDPOPolicy
    steps = args.steps if steps is None else steps
    warmup = args.warmup if warmup is None else warmup
    B = PAIRS_PER_GPU
    micro = args.micro_pairs or B
    eva = None
    if omnilmm:
        from rlaifv_b200.omnilmm_model import OmniLMMDPOPolicy, omnilmm_dims
        dims = omnilmm_dims(num_layers=args.layers)
        if not args.omnilmm_no_tower:
            from rlaifv_b200.eva_tower import EvaDims
            eva = EvaDims() if args.layers == 32 else EvaDims(depth=max(2, args.layers * 2))
            if not args.micro_pairs:
                micro = max(1, B // 2)        # whole-batch tower + decoder activations do not fit beside 12 B params
        policy = OmniLMMDPOPolicy(dims, torch.device("cuda", local_rank), seed=0, eva_dims=eva)
    else:
        dims = LlavaDims(num_layers=args.layers)
        policy = LlavaDPOPolicy(dims, torch.device("cuda", local_rank), seed=0)
    if lora:
        policy.enable_lora(r=64, alpha=16)
    engine = DPOStepEngine(policy, lr=1e-5 if lora else 5e-7, weight_decay=0.01, total_steps=2672, micro_pairs=micro,
                           rank=rank, world=world)
    # HBM plan: with the optimizer state sharded over >= 2 GPUs there is room to stash the normalised inputs
    # and the SwiGLU product (no recompute in the backward); one GPU holds the unsharded 81 GB state.
    policy.stash_extra = world > 1 and not args.no_stash_extra and not (omnilmm and eva is not None)
    # one GPU, full fine-tuning: room for the SwiGLU product only (peak ~172 of 180 GB); OOM falls back below
    policy.stash_act = world == 1 and not lora and not omnilmm and not args.no_stash_extra
    T = PROMPT_LEN + RESP_LEN - 1 + (dims.num_query + 2 if omnilmm else dims.num_patches)

    def make_host_batch(s):
        if not omnilmm:
            return synthetic_batch(rank, s, B)
        hb = synthetic_omni_batch(rank, s, B, dims)
        if eva is not None:                   # the whole config (d): pixels in, 448 px
            g = torch.Generator().manual_seed(4321 + 1000 * rank + s)
            hb["images"] = torch.randn(B, 3, eva.img_size, eva.img_size, generator=g).pin_memory()
        return hb

    # frozen-reference log-probs = initial policy log-probs (step-0 loss = ln 2 known answer)
    host_batches = [make_host_batch(s) for s in range(2)]
    for hb in host_batches:
        rw, rr = [], []
        for lo in range(0, B, micro):
            hi = min(B, lo + micro)
            ids = torch.cat([hb["concatenated_input_ids"][lo:hi], hb["concatenated_input_ids"][B + lo:B + hi]])
            lab = torch.cat([hb["concatenated_labels"][lo:hi], hb["concatenated_labels"][B + lo:B + hi]])
            out = policy.forward_logps(ids, lab, hb["images"][lo:hi], keep_stash=False)
            rw.append(out["logp"][: hi - lo].float().cpu())
            rr.append(out["logp"][hi - lo:].float().cpu())
        hb["ref_win_logp"] = torch.cat(rw).pin_memory()
        hb["ref_rej_logp"] = torch.cat(rr).pin_memory()
    dev_batches = [{k: (v.cuda(local_rank) if torch.is_tensor(v) else v) for k, v in hb.items()} for hb in host_batches]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    loss_host = torch.zeros(9, dtype=torch.float32).pin_memory()

    def run_steps(batches, n, read_back):
        m = None
        for s in range(n):
            m = engine.train_step(batches[s % len(batches)])
            if read_back:
                loss_host.copy_(m, non_blocking=True)
                torch.cuda.current_stream().synchronize()
        engine.opt.wait_all()      # the last step's parameter all-gathers belong to the timed region
        return m

    try:
        step0 = engine.train_step(dev_batches[0], optimizer_step=False)   # known-answer check (no update)
        loss0 = float(step0[0].item())
    except torch.OutOfMemoryError:
        # whole-batch activations did not fit next to the optimizer state: fall back to smaller micro-batches
        policy._stash = None
        policy._bufs.clear()
        torch.cuda.empty_cache()
        if policy.stash_act:
            policy.stash_act = False            # first give back the optional stash, keep the whole-batch pass
        else:
            policy.stash_extra = False
            micro = max(1, micro // 2)
            engine.micro_pairs = micro
        step0 = engine.train_step(dev_batches[0], optimizer_step=False)
        loss0 = float(step0[0].item())

    # ---- device-resident timing (value) ----
    run_steps(dev_batches, warmup, False)
    sampler = ClockSampler(local_rank)
    launches0 = lib.launch_count()
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t_host0 = time.perf_counter()
    last_metrics = run_steps(dev_batches, steps, False)
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / steps   # CPU time to enqueue one step
    e1.record()
    barrier()
    ms_dev = e0.elapsed_time(e1) / steps
    launches = (lib.launch_count() - launches0) // max(1, steps)
    if dump_dir and rank == 0:          # before the e2e steps below move the parameters on
        dump_outputs(dump_dir, last_metrics, policy)
    # ---- end-to-end timing through the public call with host buffers (e2e) ----
    run_steps(host_batches, 1, True)
    barrier()
    e0.record()
    run_steps(host_batches, steps, True)
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1) / steps
    clocks = sampler.stop()
    t = torch.tensor([ms_dev, ms_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = t.tolist()

    # ---- roofline of the dominant kernel: every GEMM launch of one instrumented step ----
    gemm_events = []
    orig_gemm = ops.gemm

    def timed_gemm(a, b, out=None, **kw):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        r = orig_gemm(a, b, out, **kw)
        e.record()
        K = a.shape[0] if kw.get("a_mn") else a.shape[1]
        gemm_events.append((s, e, 2.0 * r.shape[0] * r.shape[1] * K))
        return r

    orig_dual = ops.gemm_dual

    def timed_dual(a, b, a2, b2, out, **kw):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        r = orig_dual(a, b, a2, b2, out, **kw)
        e.record()
        gemm_events.append((s, e, 2.0 * r.shape[0] * r.shape[1] * (a.shape[1] + kw["k2"])))
        return r

    adamw_events = []
    orig_adamw = ops.adamw_step

    def timed_adamw(master, *a, **kw):
        st = torch.cuda.current_stream()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(st)
        orig_adamw(master, *a, **kw)
        e.record(st)
        adamw_events.append((s, e, 28.0 * master.numel()))   # fp32 p,m,v read+write, bf16 grad read, bf16 param write

    import rlaifv_b200.zero2 as _z
    ops.gemm = timed_gemm
    ops.gemm_dual = timed_dual
    _z.ops.adamw_step = timed_adamw
    try:
        engine.train_step(dev_batches[0])
        torch.cuda.synchronize()
    finally:
        ops.gemm = orig_gemm
        ops.gemm_dual = orig_dual
        _z.ops.adamw_step = orig_adamw
    hbm_peak = 6572.2
    pk = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        with open(pk) as f:
            hbm_peak = json.load(f).get("hbm_gbs", hbm_peak)
    big = [(s, e, b) for s, e, b in adamw_events if b > 1e9]     # the per-layer buckets (5.7 GB each)
    adamw_gbs = (sum(b for _, _, b in big) / (sum(s.elapsed_time(e) for s, e, _ in big) * 1e-3) / 1e9) if big else None
    gemm_ms = sum(s.elapsed_time(e) for s, e, _ in gemm_events)
    gemm_flops = sum(f for _, _, f in gemm_events)
    peak_sus, peak_burst, peak_kind = measured_peaks()
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12
    # DRAM traffic of the dominant kernel: NOT measured in this run — read from the committed `ncu --set full` capture
    # (bytes per launch of the forward qkv GEMM; the same capture lists dgrad / wgrad) — profiles/ncu_gemm_traffic.json
    traffic, traffic_note = None, None
    tp = os.path.join(REPO, "profiles", "ncu_gemm_traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            tj = json.load(f)["gemm"][0]
        traffic = tj["dram_bytes_per_launch"]
        traffic_note = "from profiles/ncu_gemm_traffic.json (ncu --set full, not measured in this run): %s: %.3g B DRAM " \
                       "per launch vs %.3g B algorithmic" % (tj["launch"], tj["dram_bytes_per_launch"],
                                                             tj["algorithmic_bytes"])

    total_pairs = B * world
    value = total_pairs / (ms_dev * 1e-3)
    e2e_value = total_pairs / (ms_e2e * 1e-3)
    hb = host_batches[0]
    h2d = sum(v.numel() * v.element_size() for v in hb.values() if torch.is_tensor(v))
    f_pair = omni_flops_per_pair(dims, T) if omnilmm else flops_per_pair(T)
    if omnilmm and eva is not None:
        f_pair += 3 * eva_flops_per_image(eva)             # trainable tower: fwd + bwd = 3 x fwd, one image per pair
    if lora:   # BASELINE.md §3 config (e): base wgrad skipped, adapters (159 907 840 params) added
        n_dec = 32 * (4 * 4096 ** 2 + 3 * 4096 * 11008)
        n_head = 4096 * 32000
        attn_seq = 32 * 4 * T * T * 4096 * 0.5
        f_clip = 2 * 23 * (4 * 1024 ** 2 + 2 * 1024 * 4096) * 577 + 23 * 4 * 577 ** 2 * 1024 + 2 * 588 * 1024 * 576
        f_proj = 2 * (1024 * 4096 + 4096 ** 2) * 576
        f_pair = 2 * T * (4 * (n_dec + n_head) + 6 * 159907840) + 3 * 2 * attn_seq + f_clip + 3 * f_proj
    if omnilmm:
        wl = ("OmniLMM-12B (RLAIF-V-12B) DPO bf16: EVA tower 448px (63 blocks, trainable) + resampler + Mistral-7B GQA "
              "decoder, %d pairs/GPU, 512-tok responses (T=%d), ZeRO-2 AdamW" % (B, T)) if eva is not None else \
             ("OmniLMM-12B DPO DOWNSTREAM OF THE VISION TOWER (resampler + Mistral-7B GQA decoder) bf16, %d pairs/GPU, "
              "1024 vision tokens, 512-tok responses (T=%d), ZeRO-2 AdamW" % (B, T))
        metric = "preference-pairs/sec OmniLMM-12B DPO step" + ("" if eva is not None else " (downstream of the vision tower)")
    else:
        wl = "LLaVA-1.5-7B %sDPO bf16, %d pairs/GPU, 336px, 512-tok responses (T=%d), ZeRO-2 AdamW" % (
            "LoRA(r=64)-" if lora else "", B, T)
        metric = "preference-pairs/sec LLaVA-1.5-7B %sDPO step" % ("LoRA-" if lora else "")
    line = {
        "metric": metric, "value": value, "unit": "pairs/s",
        "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_dev,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": wl,
                   "layers": args.layers, "pairs_per_gpu": B, "micro_pairs": micro, "parallelism": "dp%d" % world,
                   "stash_extra": bool(policy.stash_extra), "stash_act": bool(policy.stash_act),
                   "compact_head": bool(policy.compact_head),
                   "l2": "per-step working set (>100 GB of weights/activations) is far larger than the 126 MB L2",
                   "step0_loss": loss0, "step0_loss_expected": math.log(2.0)},
        "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 36,
                "ms_per_step": ms_e2e},
        "hbm_peak_gb": torch.cuda.max_memory_allocated() / 2 ** 30,
        "gpu_launches": int(launches), "host_enqueue_ms_per_step": host_enqueue_ms,
        "host_enqueue_note": "wall time of the enqueue loop INCLUDING blocking on the full launch queue; the real host "
                             "work is ~12 us per launch (profiles/r02_host_overhead.log: 13 ms per step)",
        "clocks": clocks,
        "model_flops_per_pair": f_pair,
        "step_tflops_per_gpu": value / world * f_pair / 1e12,
        "step_frac_of_peak": {"measured_sustained_%g" % peak_sus: value / world * f_pair / 1e12 / peak_sus,
                              "measured_burst_%g" % peak_burst: value / world * f_pair / 1e12 / peak_burst,
                              "datasheet_2250": value / world * f_pair / 1e12 / 2250.0},
        "roofline": {"bound": "tensor", "kernel": "gemm2_bf16_kernel / gemm_bf16_kernel (tcgen05, all GEMM launches of a step)", "achieved": achieved,
                     "peak": peak_sus, "unit": "TFLOP/s", "frac": achieved / peak_sus, "traffic": traffic, "traffic_note": traffic_note,
                     "peak_source": "%s bf16_tflops_sustained (kernel timed inside a long step); burst %g"
                                    % (peak_kind, peak_burst),
                     "frac_of_burst": achieved / peak_burst,
                     "frac_note": "the sustained figure is a cuBLAS 8192^3 matmul run back to back under the same power "
                                  "cap — a library measurement, not a hardware bound, so frac can exceed 1 when this "
                                  "kernel moves fewer bytes per FLOP; frac_of_burst relates it to the same matmul timed alone",
                     "gemm_launches": len(gemm_events), "gemm_ms_per_step": gemm_ms,
                     "gemm_share_of_step": gemm_ms / ms_dev},
        "roofline_hbm": {"bound": "hbm", "kernel": "adamw_kernel (fused AdamW on a 202M-parameter layer bucket)",
                         "achieved": adamw_gbs, "peak": hbm_peak, "unit": "GB/s",
                         "frac": (adamw_gbs / hbm_peak) if adamw_gbs else None,
                         "note": "28 algorithmic bytes per parameter; timed on the optimizer side stream while the "
                                 "backward's GEMMs run concurrently"},
    }
    # release everything this workload holds (the next workload / the checker legs need the HBM)
    policy._stash = None
    policy._bufs.clear()
    engine.opt.wait_all()
    torch.cuda.synchronize()
    del engine, policy, dev_batches, host_batches
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    return line


EXTRA_KEYS = ("metric", "value", "unit", "ms_per_step", "steps", "warmup", "e2e", "gpu_launches", "hbm_peak_gb",
              "model_flops_per_pair", "step_tflops_per_gpu", "step_frac_of_peak", "config")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--micro-pairs", type=int, default=0, help="pairs per micro-batch (0 = auto)")
    ap.add_argument("--layers", type=int, default=32, help="debug only; anything but 32 is not the benchmark")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stash-extra", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the `extra` sub-records (configs e and d)")
    ap.add_argument("--lora", action="store_true", help="BASELINE config (e): LoRA-DPO r=64 as the (only) workload")
    ap.add_argument("--omnilmm", action="store_true",
                    help="BASELINE config (d) as the (only) workload: EVA tower + resampler + Mistral-7B GQA decoder "
                         "(11.6 B trainable parameters: needs >= 2 GPUs for the ZeRO-2 sharded fp32 optimizer state)")
    ap.add_argument("--omnilmm-no-tower", action="store_true",
                    help="with --omnilmm: feed the tower's output tokens (the round-1 boundary; fits one GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/*.npy (see dump_outputs), so that two builds "
                         "can be compared on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    line = run_workload(args, rank, local_rank, world, lora=args.lora, omnilmm=args.omnilmm, dump_dir=args.dump_outputs)
    headline = not (args.lora or args.omnilmm)
    if headline and not args.no_extras:
        # BASELINE configs (e) and (d) as sub-records of the same run, with the same --steps / --warmup.
        # Every rank runs them (collectives inside); a failure is recorded, never raised.
        extra = {}
        plan = [("lora_dpo_config_e", dict(lora=True, omnilmm=False))]
        if world >= 2:
            plan.append(("omnilmm_12b_config_d", dict(lora=False, omnilmm=True)))
        else:
            extra["omnilmm_12b_config_d"] = {
                "unavailable": "11.6 B trainable parameters x 16 B (bf16 param + grad, fp32 master/m/v) = 186 GB do not "
                               "fit one 180 GB GPU; measured at N >= 2 (ZeRO-2 shards the 139 GB optimizer state)"}
        for name, kw in plan:
            try:
                sub = run_workload(args, rank, local_rank, world, extras=True, **kw)
                extra[name] = {k: sub[k] for k in EXTRA_KEYS if k in sub}
            except Exception as exc:                       # noqa: BLE001 - the headline line must survive
                extra[name] = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:300])}
                torch.cuda.empty_cache()
        line["extra"] = extra
    if rank == 0:
        if headline and not args.no_cpu_baseline and world == 1:
            line["parity_full_width"] = full_width_parity_report()
            v, cores, kind, sample, timings = cpu_reference_pairs_per_sec(reps=2, warmup=1)
            line["cpu_baseline"] = {"value": v, "unit": "pairs/s", "cores": cores, "kind": kind, "sample": sample,
                                    "timings": timings}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
