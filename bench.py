#!/usr/bin/env python
"""bench.py — (region,token) pairs/s, forward+backward, of the ViLBERT two-stream hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--config 2|3|4|5]   # this repo's CUDA engine
    python bench.py --impl reference --steps K --warmup W               # CPU arm (reference algorithm on the host cores)
    torchrun ... bench.py --gpus N ...                                   # one rank per GPU, pure data parallel

Workloads = BASELINE.json configs[1..4] (per-GPU share of the global batch, synthetic inputs of the named shapes):
  --config 2 (default, the headline metric)  bert_base_6layer_6conect, B=64, 100 regions x 36 tokens, VQA BCE objective
  --config 3  bert_base_6layer_6conect, B=64 (global 512 / 8), 37 regions (36 + global) x 36 tokens, the three-loss
              pre-training objective of BertForMultiModalPreTraining (masked-LM CE + masked-region KL + alignment CE)
  --config 4  bert_large_6layer_6conect, B=32 (global 256 / 8), 100 regions x 60 tokens, VL-logit CE over 4 options (VCR)
  --config 5  one 12-in-1 multi-task iteration (tasks 1-2-4-7-8-9-10-11-12-13-15-17 of vilbert_tasks.yml at batch / 8,
              task tokens on): 12 forward+backward passes of different shapes and objectives per step
One "step" = train-mode forward (every nn.Dropout of the reference active, in-kernel masks) of the encoder and ALL heads (as
VILBertForVLTasks.forward always computes them), the task objective, backward of everything with a gradient path and, for
N > 1, the gradient all-reduce. The optimizer is not part of the named metric (SURVEY.md §8d): the fused AdamW (which also
rewrites the 16-bit weight copies and zeroes the gradients, so the step itself has no cast / memset) is timed in the same run
and reported separately as `optimizer` / `train_step`.

`value` is measured with inputs resident in HBM (CUDA-graph replay); `e2e` runs the same step from pinned HOST buffers
through the engine API (H2D of the batch and D2H of the loss inside the timed region). Prints ONE JSON line.

`--dump-outputs DIR` writes what the last timed step returned (outputs, loss and parameter gradient of every plan) to DIR as
.npy files. Inputs and weights are seeded, so two builds run with the same arguments can be compared array by array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "(region,token) pairs/sec fwd+bwd, bert_base_6layer_6conect"
# 12-in-1 mix: (task, global batch of vilbert_tasks.yml, regions, tokens, objective). Retrieval expands to 4 options per
# caption (task_utils.py:186-246), NLVR2 to 2 images per sample (:289-310); V-logit-mc tasks (Visual7w, GuessWhat) drive the
# vision_logit head like V-logit (their gather over <= 204 choice ids is not modelled: same kernels, same bytes).
TASKS_12IN1 = [("TASK1", 128, 101, 23, "vqa"), ("TASK2", 128, 101, 26, "vqa"), ("TASK4", 256, 200, 20, "vlogit_bce"),
               ("TASK7", 512, 101, 30, "logit_ce"), ("TASK8", 512, 101, 30, "logit_ce"), ("TASK9", 256, 101, 20, "vlogit_bce"),
               ("TASK10", 256, 101, 20, "vlogit_bce"), ("TASK11", 256, 101, 20, "vlogit_bce"), ("TASK12", 128, 101, 40, "binary_ce"),
               ("TASK13", 256, 101, 56, "tri_ce"), ("TASK15", 128, 101, 26, "gqa"), ("TASK17", 64, 306, 256, "vlogit_bce")]
CONFIGS = {
    2: dict(model="bert_base_6layer_6conect", tasks=[("VQA", 64, 100, 36, "vqa")], task_tokens=False, per_gpu=True,
            what="VQA-shape synthetic: per-GPU batch 64, 100 regions x 2048 feats, 36 tokens, all heads + VQA BCE loss"),
    3: dict(model="bert_base_6layer_6conect", tasks=[("CC", 64, 37, 36, "pretraining")], task_tokens=False, per_gpu=True, heads="pretraining",
            what="Conceptual-Captions-shape synthetic: per-GPU batch 64 (global 512 / 8), 36 + 1 regions, 36 tokens, masked-LM CE + masked-region KL + alignment CE"),
    4: dict(model="bert_large_6layer_6conect", tasks=[("VCR", 32, 100, 60, "logit_ce")], task_tokens=False, per_gpu=True,
            what="VCR-shape synthetic: bert_large, per-GPU batch 32 (global 256 / 8 = 8 questions x 4 options), 100 regions, 60 tokens, VL-logit CE"),
    5: dict(model="bert_base_6layer_6conect", tasks=TASKS_12IN1, task_tokens=True, per_gpu=False,
            what="12-in-1 multi-task iteration (tasks 1-2-4-7-8-9-10-11-12-13-15-17, vilbert_tasks.yml batch / 8 per GPU, task tokens): 12 fwd+bwd passes per step"),
}


def load_config_json(name):
    with open(os.path.join(ROOT, "vilbert-multi-task_b200", "configs", name + ".json")) as f:
        return json.load(f)


def algorithmic_flops_fwd(c, Nv, Nt):
    """Closed form of SURVEY.md §8d (2 FLOP per MAC, forward, per sample, heads included)."""
    Ht, It, Hv, Iv, Hb, Fv, V = c["hidden_size"], c["intermediate_size"], c["v_hidden_size"], c["v_intermediate_size"], c["bi_hidden_size"], c["v_feature_size"], c["vocab_size"]
    Lt, Lv, Lc = c["num_hidden_layers"], c["v_num_hidden_layers"], len(c["v_biattention_id"])
    f_text = 2 * Nt * (4 * Ht * Ht + 2 * Ht * It) + 4 * Nt * Nt * Ht
    f_vis = 2 * Nv * (4 * Hv * Hv + 2 * Hv * Iv) + 4 * Nv * Nv * Hv
    f_conn = 2 * (3 * Nv * Hv * Hb + 3 * Nt * Ht * Hb + Nv * Hb * Hv + Nt * Hb * Ht + 2 * Nv * Hv * Iv + 2 * Nt * Ht * It) + 8 * Nt * Nv * Hb
    f_emb = 2 * Nv * (Fv + 5) * Hv
    f_pool = 2 * (Ht + Hv) * Hb
    f_heads = 2 * (Nt * (Ht * Ht + Ht * V) + Nv * (Hv * Hv + Hv * c["v_target_size"]) + 2 * Hb + Hb * 2 * Hb + 2 * Hb * 3129 + Hb * 2 * Hb
                   + 2 * Hb * 1533 + 0.5 * (2 * Hb * 2 * Hb + 2 * Hb * 2) + Hb * 4 + Nv * Hv + Nt * Ht)
    return Lt * f_text + Lv * f_vis + Lc * f_conn + f_emb + f_pool + f_heads


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1425.6), d.get("bf16_tflops", 1650.9), d.get("hbm_gbs", 6575.1), "measured (MEASURED_PEAKS.json)"
    return 1400.0, 1590.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe). The sampler
    is started before the warm-up (nvidia-smi needs a moment to come up); only samples whose timestamp falls inside the
    marked window are used (all samples if none does)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def start(self):
        q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        self.t.join(timeout=2)
        rows = [r for (ts, r) in self.rows if self.t0 is not None and self.t0 - 0.05 <= ts <= (self.t1 or ts) + 0.1]
        window = "timed region"
        if not rows:
            rows, window = [r for (_, r) in self.rows], "whole run (no sample fell inside the timed region)"
        num = lambda x: x.replace(".", "", 1).isdigit()
        sm = sorted(int(float(r[1])) for r in rows if len(r) > 1 and num(r[1]))
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 4 + i and r[4 + i].lower().startswith("active") for r in rows)]
        mx = [int(float(r[2])) for r in rows if len(r) > 2 and num(r[2])]
        pw = [float(r[3]) for r in rows if len(r) > 3 and num(r[3])]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None, "reasons": reasons,
                "samples": len(sm), "power_w_max": max(pw) if pw else None, "window": window}


# ---------------------------------------------------------------------------------------------- CPU arm
def run_cpu_reference(cfgj, B, Nv, Nt, steps, warmup, budget_s=None, threads=None):
    """The reference algorithm's VILBertForVLTasks fwd + VQA loss + bwd, fp32, on the host cores, at a FIXED sample batch B:
    `warmup` untimed steps (>= 1, so that allocator / thread-pool start-up never lands in a timed step), then `steps` timed
    steps, fewer only if `budget_s` seconds have passed. Runs the oracle port (kind "port"), which tests/test_oracle_golden.py
    holds bit-exact to the reference's recorded outputs and gradients on CPU."""
    import torch
    from oracle import vilbert_oracle as O
    if threads is None:
        try:
            usable = len(os.sched_getaffinity(0))
        except AttributeError:
            usable = os.cpu_count() or 1
        threads = int(os.environ.get("VB_CPU_THREADS", min(usable, 32)))
    torch.set_num_threads(threads)
    cfg = O.make_config(cfgj)
    P = O.synth_params(cfg, seed=0)
    inp = O.synth_inputs(cfg, B, Nv, Nt, seed=1234)
    tgt = O.synth_vqa_target(B, 3129)
    Pg = {k: v.clone().requires_grad_(True) for k, v in P.items() if k != "cls.predictions.decoder.weight"}
    Pg["cls.predictions.decoder.weight"] = Pg["bert.embeddings.word_embeddings.weight"]

    def one_step():
        t0 = time.perf_counter()
        for v in Pg.values():
            v.grad = None
        _, heads = O.vilbert_for_vl_tasks(Pg, cfg, inp["input_txt"], inp["input_imgs"], inp["image_loc"], inp["token_type_ids"], inp["attention_mask"],
                                          inp["image_attention_mask"], inp["co_attention_mask"], inp["task_ids"])
        O.vqa_loss(heads[0], tgt).backward()
        return time.perf_counter() - t0

    t_start = time.perf_counter()
    for _ in range(max(warmup, 1)):
        one_step()
    times = []
    for _ in range(steps):
        times.append(one_step())
        if budget_s is not None and time.perf_counter() - t_start > budget_s:
            break
    sec = sum(times) / len(times)
    return dict(value=B * Nv * Nt / sec, unit="pairs/s", cores=threads, kind="port", sec_per_step=sec, sample_batch=B, steps_timed=len(times),
                sample=f"oracle port (bit-exact vs the reference on CPU): VILBertForVLTasks fwd + VQA loss + "
                       f"bwd, fp32, fixed B={B} x {Nv} regions x {Nt} tokens, {max(warmup, 1)} warm-up + {len(times)} timed step(s), {threads} threads")


# ---------------------------------------------------------------------------------------------- synthetic targets
def synth_loss_inputs(plan, kind, seed, torch):
    """Host tensors for the static label / target inputs of a plan's fused objective (SURVEY.md §8d 'Targets')."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    if kind in ("vqa", "gqa"):
        n = 3129 if kind == "vqa" else 1533
        t = torch.zeros(plan.B, n)
        idx = torch.randint(0, n, (plan.B, 3), generator=g)
        t.scatter_(1, idx, torch.tensor([0.3, 0.6, 0.9, 1.0])[torch.randint(0, 4, (plan.B, 3), generator=g)])
        out["vqa_target" if kind == "vqa" else "target"] = t
    elif kind == "vlogit_bce":
        out["target"] = (torch.rand(plan.B, plan.Nv, generator=g) < 0.05).float()
    elif kind in ("logit_ce", "binary_ce", "tri_ce"):
        rows, hi = {"logit_ce": (plan.B // 4, 4), "binary_ce": (plan.B // 2, 2), "tri_ce": (plan.B, 3)}[kind]
        out["labels"] = torch.randint(0, hi, (rows,), generator=g)
    elif kind == "pretraining":
        lm = torch.full((plan.B * plan.Nt,), -1, dtype=torch.long)
        sel = torch.rand(plan.B * plan.Nt, generator=g) < 0.15
        lm[sel] = torch.randint(0, plan.cfg.vocab_size, (int(sel.sum()),), generator=g)
        out["masked_lm_labels"] = lm
        il = torch.full((plan.B, plan.Nv - 1), -1, dtype=torch.long)
        il[torch.rand(plan.B, plan.Nv - 1, generator=g) < 0.15] = 1
        il[:, 0] = 1
        out["image_label"] = il
        out["image_target"] = torch.softmax(torch.randn(plan.B, plan.Nv - 1, plan.cfg.v_target_size, generator=g), -1)
        out["next_sentence_label"] = torch.randint(0, 2, (plan.B,), generator=g)
    return out


DUMP_BYTES = 60 * 2 ** 20    # all arrays of --dump-outputs together, leaving room for the .npy headers below 64 MB


def dump_outputs(out_dir, T, eng, torch):
    """What the timed step hands its caller after the last run, as float32 .npy files: every output of each plan
    (`<task>.<output>.npy`), its loss (`<task>.loss.npy`) and the flat fp32 parameter gradient (`param_grad.npy`, accumulated over
    every step of the run). An array larger than its equal share of DUMP_BYTES is replaced by a 1-D sample of it, at sorted
    flat indices drawn from a CPU generator seeded with 0, so the same arguments select the same elements on every build.
    With a shared activation arena only the plan that ran last still holds its outputs; the others contribute their loss."""
    import numpy as np
    arrays = {}
    for t in T:
        plan = t["plan"]
        if eng.arena is None or eng.arena_owner[0] is plan:
            for name, x in plan.outputs.items():
                arrays[f"{t['name']}.{name}"] = x
        arrays[f"{t['name']}.loss"] = plan.loss
    arrays["param_grad"] = eng.ps.grad
    cap = DUMP_BYTES // 4 // len(arrays)
    os.makedirs(out_dir, exist_ok=True)
    for name, x in arrays.items():
        x = x.detach()
        if x.numel() > cap:
            idx = torch.randint(0, x.numel(), (cap,), generator=torch.Generator().manual_seed(0)).sort().values
            x = x.reshape(-1)[idx.to(x.device)]
        np.save(os.path.join(out_dir, name + ".npy"), x.float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--precision", default="fp16", choices=["fp16", "fp32", "bf16"],
                    help="operand precision: fp16 forward / bf16 gradient operands (default), split-precision fp32 parity mode, all-bf16")
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch of a single-task config")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="N > 1: all-reduce after the whole backward instead of overlapping it")
    ap.add_argument("--ddp-mode", default="pieces", choices=["graph", "pieces"],
                    help="N > 1 overlapped step: 'pieces' (default) = one graph per backward piece, collectives issued from the host between "
                         "them; 'graph' = ONE CUDA graph per step with the NCCL all-reduces captured on a side stream (measured 0.6 %% faster at "
                         "N = 2, but ProcessGroupNCCL's watchdog hangs at teardown while captured collectives are alive: opt-in)")
    ap.add_argument("--nccl-max-ctas", type=int, default=0, help="N > 1: cap NCCL's CTAs per collective (NCCL_MAX_CTAS) so that the all-reduce "
                                                                  "overlapping the backward takes fewer SMs from the persistent GEMMs; 0 = NCCL default")
    ap.add_argument("--bwd-gemm-ctas", type=int, default=-1,
                    help="N > 1: persistent CTAs of the backward-pass GEMMs (they run beside NCCL's all-reduce kernels; a GEMM CTA that finds "
                         "its SM taken starts after the others and serialises its whole static tile share). -1 = 132 (measured at N = 2: 12.39 ms/step vs "
                         "12.49 with one CTA per SM and 12.46 with 116), 0 = one per SM")
    ap.add_argument("--arena-gb", type=float, default=0.0,
                    help="share ONE activation arena of this size between the plans (Engine.enable_activation_arena): config 5 keeps 12 plans "
                         "whose private activations add up to 42.7 GB; 0 = private buffers per plan")
    ap.add_argument("--segments", type=int, default=8, help="N > 1: number of backward pieces whose gradient ranges are all-reduced while the rest runs")
    ap.add_argument("--eval-mode", action="store_true", help="disable the dropout layers (reference eval mode); default is train mode")
    ap.add_argument("--legacy-prologue", action="store_true", help="round-1 step body: weight cast + gradient memset inside the step, no fused optimizer")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-module-api", action="store_true", help="skip the VILBertForVLTasks.forward -> loss.backward() leg")
    ap.add_argument("--cpu-batch", type=int, default=8)
    ap.add_argument("--profile-ops", action="store_true", help="print the per-kernel-class time table to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs, loss and parameter gradient of the last timed step to DIR "
                                                          "as float32 .npy files (a fixed sample of each large array; rank 0)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    C = CONFIGS[a.config]
    cfgj = load_config_json(C["model"])
    if C["task_tokens"]:
        cfgj = dict(cfgj, task_specific_tokens=True)
    tasks = []
    for (tname, gb, Nv, Nt, kind) in C["tasks"]:
        b = gb if C["per_gpu"] else gb // 8
        if a.batch and len(C["tasks"]) == 1:
            b = a.batch
        tasks.append((tname, b, Nv, Nt, kind))
    workload = f"config {a.config}: {C['model']} {C['what']}, fwd+bwd"

    if a.impl == "reference":
        if rank != 0:
            return
        W = max(min(a.warmup, 2), 1)
        c2 = load_config_json("bert_base_6layer_6conect")
        r = run_cpu_reference(c2, a.cpu_batch, 100, 36, a.steps, W)
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "pairs/s", "n_gpus": a.gpus, "steps": r["steps_timed"], "warmup": W,
                          "ms_per_step": r["sec_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic", "config": {"workload": "config 2: bert_base_6layer_6conect VQA-shape synthetic, 100 regions x 36 tokens, all heads + VQA BCE loss, fwd+bwd",
                                     "sample_batch": r["sample_batch"],
                                     "note": "CPU arm on the host cores of rank 0 (no GPU work whatever --gpus says): a fixed B=8 sample of the workload per step "
                                             "(per-sample cost is batch-independent on CPU at this size)"},
                          "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
                          "e2e": {"value": r["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    import torch.distributed as dist
    from vilbert_b200.config import BertConfig
    from vilbert_b200.engine import Engine, LOSS_HEADS
    from vilbert_b200.optim import FusedAdamW
    from oracle import vilbert_oracle as O   # synthetic-input generator + cpu_baseline leg only

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and a.nccl_max_ctas > 0:
        os.environ.setdefault("NCCL_MAX_CTAS", str(a.nccl_max_ctas))
    if world > 1:
        # NCCL prints its version banner on stdout; keep stdout for the single JSON line
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    if world > 1:
        # a collective that never completes must not hold the box until the caller's limit: give up loudly after 15 minutes
        wd = threading.Timer(900.0, lambda: (print(f"[bench] rank {rank}: watchdog: no result after 900 s, aborting", file=sys.stderr), os._exit(3)))
        wd.daemon = True
        wd.start()
    W = max(a.warmup, 3)
    cfg_o = O.make_config(cfgj)
    eng = Engine(BertConfig.from_dict(cfgj), dev, heads=C.get("heads", "vl"), precision=a.precision)
    if world > 1:
        eng.bwd_gemm_max_ctas = a.bwd_gemm_ctas if a.bwd_gemm_ctas >= 0 else 132
    if a.arena_gb > 0:
        eng.enable_activation_arena(int(a.arena_gb * 2 ** 30))
    # random-init weights of the named architecture (reference init: N(0, 0.02), zero bias, LN 1/0); same seed on every rank
    g = torch.Generator(device=dev).manual_seed(0)
    eng.ps.flat.normal_(0.0, 0.02, generator=g)
    for name in eng.ps.entries:
        if "LayerNorm" in name or ".logit_fc.2." in name:
            eng.ps.p(name).fill_(1.0 if name.endswith("weight") else 0.0)
        elif name.endswith(".bias"):
            eng.ps.p(name).zero_()
    eng.refresh_weights()

    # ---------------- plans, synthetic batches (different per rank; host-pinned), optimizer
    keys = ("input_txt", "input_imgs", "image_loc", "token_type_ids", "attention_mask", "image_attention_mask")
    n_host = 4 if len(tasks) == 1 else 1
    T = []
    for ti, (tname, B, Nv, Nt, kind) in enumerate(tasks):
        plan = eng.plan(B, Nt, Nv, grad_outputs=LOSS_HEADS[kind], loss=kind, train=not a.eval_mode)
        host = []
        for i in range(n_host):
            inp = O.synth_inputs(cfg_o, B, Nv, Nt, seed=1234 + rank + 1000 * i + 17 * ti, task_id=(ti + 1) if C["task_tokens"] else None)
            host.append({k: v.pin_memory() for k, v in inp.items() if torch.is_tensor(v)})
        lin = {k: v.pin_memory() for k, v in synth_loss_inputs(plan, kind, 99 + rank + 7 * ti, torch).items()}
        plan.load_inputs(*(host[0][k] for k in keys), task_ids=host[0].get("task_ids"))
        for k, v in lin.items():
            (plan.vqa_target if k == "vqa_target" else plan.loss_inputs[k]).copy_(v.reshape((plan.vqa_target if k == "vqa_target" else plan.loss_inputs[k]).shape))
        T.append(dict(name=tname, plan=plan, host=host, kind=kind, B=B, Nv=Nv, Nt=Nt))
    torch.cuda.synchronize()
    # the reference's optimizer setup (train_tasks.py:401-426): one group per tensor, lr 1e-4 for vil_* heads, no decay on bias / LayerNorm
    class _P:   # minimal parameter objects over the flat buffer (the module surface builds nn.Parameters the same way)
        pass
    params = []
    for name in eng.ps.entries:
        t = torch.nn.Parameter(eng.ps.p(name), requires_grad=True)
        no_decay = any(nd in name for nd in ("bias", "LayerNorm.bias", "LayerNorm.weight"))
        params.append({"params": [t], "lr": 1e-4 if "vil_" in name else 4e-5, "weight_decay": 0.0 if no_decay else 0.01})
    opt = None if a.legacy_prologue else FusedAdamW(params, lr=4e-5, correct_bias=False, engine=eng)
    for t in T:
        if a.legacy_prologue:
            t["plan"].enable_training_prologue()
        elif t["plan"].train:
            t["plan"].prologue = [(t["plan"].lib.vb_step_counter_bump, (eng.drop_step.data_ptr(),), 0)]
    from vilbert_b200.ddp import FlatGradAllReducer
    reducer = FlatGradAllReducer(eng.ps.grad, n_buckets=8)   # NCCL all-reduce (AVG) of the flat fp32 gradient buffer
    single = len(T) == 1
    overlapped = world > 1 and single and not a.no_graph and not a.no_overlap
    comm_stream = None
    ddp_graph = False
    if overlapped and a.ddp_mode == "graph":
        plan = T[0]["plan"]
        try:
            for _ in range(2):      # warm-up outside capture (lazy module loads, NCCL channel set-up for every range size)
                plan.run_step(); reducer.allreduce()
            torch.cuda.synchronize()
            plan.capture_step_ddp(reducer.allreduce_range_sync, a.segments)
            ddp_graph = True
        except Exception as e:   # noqa: BLE001
            print(f"[bench] rank {rank}: capture_step_ddp failed ({e}); falling back to per-piece graphs", file=sys.stderr)
            try:
                torch.cuda.synchronize()
            except Exception:    # noqa: BLE001
                pass
    if overlapped and not ddp_graph:
        plan = T[0]["plan"]
        for tail_cut in (True, False):
            try:
                plan.capture_segments(a.segments, tail_cut=tail_cut)
                break
            except Exception as e:   # noqa: BLE001
                print(f"[bench] rank {rank}: capture_segments({a.segments}, tail_cut={tail_cut}) failed: {e}", file=sys.stderr)
                try:
                    torch.cuda.synchronize()
                except Exception:    # noqa: BLE001
                    pass
        else:
            overlapped = False
        comm_stream = torch.cuda.Stream()
    if not overlapped and not a.no_graph:
        for t in T:
            t["plan"].capture()

    def step(with_opt=False):
        for t in T:
            plan = t["plan"]
            if ddp_graph:
                plan.run_step_ddp()
            elif overlapped:
                works = plan.run_step_overlapped(reducer.allreduce_range, comm_stream)
                for w in works:
                    if w is not None:
                        w.wait()          # the main stream waits for the collectives
            else:
                plan.run_step()
                reducer.allreduce()
            if with_opt and opt is not None:
                opt.launch()              # one optimizer step per task backward, like the reference (train_tasks.py:550)

    def timed(fn, steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    # ---------------- device-resident throughput (the named metric: fwd + loss + bwd [+ all-reduce])
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    for _ in range(W):
        step()
    torch.cuda.synchronize()
    clocks.mark_begin()
    ms = timed(lambda i: step(), a.steps)
    clocks.mark_end()
    clk = clocks.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, T, eng, torch)     # before the legs below change the weights, inputs and gradients
    ms_step = ms / a.steps
    loss_val = float(sum(t["plan"].loss.item() for t in T))
    # ---------------- the same step followed by the fused optimizer (AdamW + 16-bit weight copies + gradient zeroing in one launch)
    ms_train = ms_opt = None
    if opt is not None:
        eng.zero_grad(force=True)
        for _ in range(3):
            step(True)
        ms_train = timed(lambda i: step(True), a.steps) / a.steps
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            opt.launch()
        e1.record(); torch.cuda.synchronize()
        ms_opt = e0.elapsed_time(e1) / 10
        eng.zero_grad(force=True)

    # ---------------- end to end from pinned host memory: H2D of the next batch overlaps the current step on a copy
    # stream into a staging set, a device copy moves it into the plan's static inputs, the loss is read back every step
    copy_stream = torch.cuda.Stream()
    loss_host = torch.zeros((a.steps + W + 4) * len(T), dtype=torch.float32).pin_memory()
    h2d_bytes = 0
    for t in T:
        plan = t["plan"]
        t["stage"] = [{k: torch.empty_like(t["host"][0][k], device=dev) for k in keys} for _ in range(2)]
        t["ev_ready"] = [torch.cuda.Event() for _ in range(2)]
        t["ev_free"] = [torch.cuda.Event() for _ in range(2)]
        t["dst"] = dict(input_txt=plan.in_ids, input_imgs=plan.in_feat, image_loc=plan.in_loc, token_type_ids=plan.in_tt, attention_mask=plan.in_amask,
                        image_attention_mask=plan.in_imask)
        h2d_bytes += sum(t["host"][0][k].numel() * t["host"][0][k].element_size() for k in keys)
        for e in t["ev_free"]:
            e.record()

    def prefetch(t, i):
        s = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(t["ev_free"][s])
            for k in keys:
                t["stage"][s][k].copy_(t["host"][i % n_host][k], non_blocking=True)
            t["ev_ready"][s].record(copy_stream)

    for t in T:
        prefetch(t, 0)

    def e2e_step(i):
        s = i % 2
        cur = torch.cuda.current_stream()
        for ti, t in enumerate(T):
            plan = t["plan"]
            prefetch(t, i + 1)
            cur.wait_event(t["ev_ready"][s])
            for k in keys:
                t["dst"][k].copy_(t["stage"][s][k], non_blocking=True)
            t["ev_free"][s].record(cur)
            if ddp_graph:
                plan.run_step_ddp()
            elif overlapped:
                for w in plan.run_step_overlapped(reducer.allreduce_range, comm_stream):
                    if w is not None:
                        w.wait()
            else:
                plan.run_step()
                reducer.allreduce()
            loss_host[i * len(T) + ti].copy_(plan.loss[0], non_blocking=True)

    for i in range(2):
        e2e_step(i)
    torch.cuda.synchronize()
    for t in T:
        prefetch(t, 0)
    ms_e2e = timed(e2e_step, a.steps)
    ms_e2e_step = ms_e2e / a.steps
    mem_gb = torch.cuda.max_memory_allocated() / 2 ** 30

    # ---------------- per-kernel-class profile (eager replay with events; the GPU is held busy first so that
    # launches are queued ahead and every event pair brackets pure execution)
    prof = None
    if rank == 0:
        ops = [op for t in T for op in (t["plan"].prologue + t["plan"].fwd + t["plan"].bwd) if op[0] is not None]   # single stream, barriers dropped
        stream = torch.cuda.current_stream().cuda_stream
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in ops]
        torch.cuda._sleep(int(60e6))
        for (fn, args, _sid), (s0, s1) in zip(ops, evs):
            s0.record()
            fn(*args, stream)
            s1.record()
        torch.cuda.synchronize()
        prof = {}
        for (fn, args, _sid), (s0, s1) in zip(ops, evs):
            name = fn.__name__
            d = prof.setdefault(name, dict(ms=0.0, n=0, flops=0.0))
            d["ms"] += s0.elapsed_time(s1); d["n"] += 1
            if name == "vb_gemm_bf16":
                ga = args[0]._obj
                d["flops"] += 2.0 * ga.M * ga.N * ga.K
            elif name.startswith("vb_attention"):
                aa = args[0]._obj
                d["flops"] += 4.0 * aa.B * aa.H * aa.Nq * aa.Nk * aa.D * (2.5 if name.endswith("bwd") else 1.0)
        if a.profile_ops:
            shapes = {}
            for (fn, args, _sid), (s0, s1) in zip(ops, evs):
                if fn.__name__ == "vb_gemm_bf16":
                    ga = args[0]._obj
                    key = (ga.M, ga.N, ga.K, "A^T" if ga.a_mn_major else "A", "B^T" if ga.b_mn_major else "B", ga.act, int(bool(ga.out_f32)), int(bool(ga.out_bf16)),
                           int(bool(ga.residual)), ga.atomic_out, 1 + int(bool(ga.A_lo)) + int(bool(ga.B_lo)))
                    d = shapes.setdefault(key, [0, 0.0])
                    d[0] += 1; d[1] += s0.elapsed_time(s1)
            print("  GEMM launches by signature (M N K majors act f32 b16 res atomic passes): n, total ms, avg us, TFLOP/s", file=sys.stderr)
            for key, (n, ms_) in sorted(shapes.items(), key=lambda kv: -kv[1][1])[:32]:
                fl = 2.0 * key[0] * key[1] * key[2] * n
                print(f"    {str(key):62s} n={n:3d} {ms_:7.3f} ms {ms_ / n * 1e3:7.1f} us {fl / ms_ / 1e9:7.1f}", file=sys.stderr)
            tot = sum(d["ms"] for d in prof.values())
            for k, d in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]):
                tf = f"{d['flops'] / d['ms'] / 1e9:8.1f} TFLOP/s" if d["flops"] else ""
                print(f"  {k:26s} n={d['n']:4d} {d['ms']:8.3f} ms {100 * d['ms'] / tot:5.1f}% {tf}", file=sys.stderr)
            print(f"  eager-replay kernel time total {tot:.3f} ms vs graph step {ms_step:.3f} ms", file=sys.stderr)

    # ---------------- the drop-in module API: VILBertForVLTasks.forward -> loss -> loss.backward() (config 2, 1 GPU)
    module_api = None
    if rank == 0 and world == 1 and a.config == 2 and not a.no_module_api:
        try:
            module_api = run_module_api(cfgj, T[0], a, torch, O, timed)
        except Exception as e:   # noqa: BLE001
            module_api = {"error": repr(e)[:300]}

    if rank != 0:
        if world > 1:
            if ddp_graph:
                for t in T:
                    t["plan"].graph_step_ddp = None
                torch.cuda.synchronize()
            dist.destroy_process_group()
        return

    peak_sus, peak_burst, hbm, peak_src = measured_peaks()
    flops_step = sum(3.0 * algorithmic_flops_fwd(cfgj, t["plan"].Nv, t["plan"].Nt) * t["B"] for t in T)   # fwd+bwd = 3 x forward (SURVEY.md §8d), per GPU
    pairs = sum(t["B"] * t["plan"].Nv * t["plan"].Nt for t in T) * world
    samples = sum(t["B"] for t in T) * world
    value = pairs / (ms_step / 1e3)
    n_launch = sum(t["plan"].n_launches_step for t in T)
    out = {
        "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": a.steps, "warmup": W, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": {"fp16": "fp16", "bf16": "bf16", "fp32": "fp16x3 (split precision)"}[a.precision],
        "data": "synthetic",
        "config": {"workload": workload, "global_batch": samples, "parallelism": f"dp{world}", "cuda_graph": not a.no_graph,
                   "tasks": [dict(task=t["name"], batch=t["B"], regions=t["plan"].Nv, tokens=t["plan"].Nt, objective=t["kind"]) for t in T] if len(T) > 1 else None,
                   "allreduce": ("none (1 GPU)" if world == 1 else (f"NCCL AVG of the flat fp32 gradient buffer, {len(T[0]['plan'].segments)} tail ranges overlapped with backward"
                                                                         + (" (one CUDA graph per step, collectives captured, never-written ranges skipped)" if ddp_graph else " (one graph per backward piece)") if overlapped
                                 else "NCCL AVG of the flat fp32 gradient buffer after each backward (8 buckets)")),
                   "bwd_gemm_ctas": (eng.bwd_gemm_max_ctas or "one per SM"),
                   "activation_arena_gb": (round(max(t["plan"].arena_bytes for t in T) / 2 ** 30, 2) if eng.arena is not None else None),
                   "l2": "working set (activations + weights + grads, GBs per step) exceeds the 126 MB L2; no explicit flush",
                   "streams": "text and vision segments on two CUDA streams (parallel graph branches)" if eng.two_streams else "single stream",
                   "numerics": {"fp16": "fp16 forward tensor-core operands, bf16 gradient operands, fp32 accumulate/residual/LayerNorm/softmax",
                                "bf16": "bf16 tensor-core operands, fp32 accumulate/residual/LayerNorm/softmax",
                                "fp32": "split precision: fp16 hi+lo forward operands, 3 tensor-core passes per contraction (fp32 parity mode)"}[a.precision],
                   "mode": "eval (dropout off)" if a.eval_mode else "train: every nn.Dropout of the reference active (p=0.1, in-kernel counter-based masks, new masks each step)",
                   "step_body": ("round-1 body: dropout bump + grad memset + weight cast + fwd + loss + bwd" if a.legacy_prologue else
                                 "dropout bump + fwd + loss + bwd; the 16-bit weight copies and the gradient zeroing are part of the fused AdamW launch (timed separately: optimizer / train_step)"),
                   "loss": loss_val, "peak_memory_gb": round(mem_gb, 2), "plans": len(T)},
        "samples_per_s": samples / (ms_step / 1e3),
        "model_tflops_per_gpu": flops_step / (ms_step / 1e3) / 1e12,
        "mfu_vs_measured_sustained_bf16": flops_step / (ms_step / 1e3) / 1e12 / peak_sus,
        "gpu_launches": n_launch * a.steps,
        "clocks": clk,
        "e2e": {"value": pairs / (ms_e2e_step / 1e3), "unit": "pairs/s", "ms_per_step": ms_e2e_step, "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": 4 * len(T), "api": "Plan.run_step on pinned-host batches (double-buffered H2D on a copy stream), loss read back every step"},
    }
    if ms_train is not None:
        out["optimizer"] = {"kind": "FusedAdamW (one launch over the flat buffers: AdamW + fp16/bf16 weight copies + gradient zeroing; reference grouping: one group per tensor, correct_bias=False)",
                            "ms_per_launch": ms_opt, "launches_per_step": len(T), "included_in_value": False}
        out["train_step"] = {"ms_per_step": ms_train, "value": pairs / (ms_train / 1e3), "unit": "pairs/s", "what": "fwd + loss + bwd (+ all-reduce) + fused AdamW, same run"}
    if module_api is not None:
        out["module_api"] = module_api
    if prof:
        gm = prof["vb_gemm_bf16"]
        ach = gm["flops"] / (gm["ms"] / 1e3) / 1e12
        # dominant single kernel = the GEMM problem signature with the largest total time in one step
        sigs = {}
        for (fn, args, _sid), (s0, s1) in zip(ops, evs):
            if fn.__name__ == "vb_gemm_bf16":
                ga = args[0]._obj
                key = (ga.M, ga.N, ga.K, int(ga.a_mn_major), int(ga.b_mn_major), ga.act, int(bool(ga.residual)), int(ga.atomic_out))
                d = sigs.setdefault(key, [0, 0.0])
                d[0] += 1; d[1] += s0.elapsed_time(s1)
        dom, (dn, dms) = max(sigs.items(), key=lambda kv: kv[1][1])
        dflops = 2.0 * dom[0] * dom[1] * dom[2]
        dach = dflops / (dms / dn / 1e3) / 1e12
        traffic, traffic_src = ncu_traffic(dom)
        out["roofline"] = {"bound": "tensor",
                           "kernel": f"gemm_tcgen05_kernel M={dom[0]} N={dom[1]} K={dom[2]} (a_mn={dom[3]} b_mn={dom[4]} act={dom[5]} residual={dom[6]} "
                                     f"atomic={dom[7]}): the GEMM signature with the largest share of the step ({dn} launches, {dms:.3f} ms)",
                           "achieved": dach, "peak": peak_sus, "unit": "TFLOP/s", "frac": dach / peak_sus,
                           "traffic": traffic, "traffic_unit": "bytes/launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, cold cache)", "traffic_source": traffic_src,
                           "algorithmic_flops_per_launch": dflops, "avg_launch_us": dms / dn * 1e3,
                           "peak_source": peak_src + ", sustained cuBLAS bf16",
                           "how": "algorithmic 2MNK / mean CUDA-event duration of that launch in an eager single-stream replay of the step"}
        out["roofline_all_gemm"] = {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (all launches of one step)",
                           "how": "sum of algorithmic 2MNK over the step's GEMM launches / sum of their CUDA-event durations in an eager single-stream replay "
                                  "(each launch bracketed by events, so launch gaps and event latency count against the kernel)",
                           "achieved": ach, "peak": peak_sus,
                           "unit": "TFLOP/s", "frac": ach / peak_sus, "traffic": None, "peak_source": peak_src + ", sustained cuBLAS bf16",
                           "launches_per_step": gm["n"], "kernel_ms_per_step": gm["ms"], "algorithmic_flops_per_step": gm["flops"],
                           "share_of_step": gm["ms"] / sum(d["ms"] for d in prof.values())}
        out["kernel_classes_ms"] = {k: round(d["ms"], 4) for k, d in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}
    if not a.no_cpu_baseline:
        c2 = load_config_json("bert_base_6layer_6conect")
        r = run_cpu_reference(c2, a.cpu_batch, 100, 36, steps=3, warmup=1, budget_s=45.0)
        out["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(out))
    sys.stdout.flush()
    if world > 1:
        if ddp_graph:      # captured collectives must be gone before the process group is torn down (else its watchdog hangs)
            for t in T:
                t["plan"].graph_step_ddp = None
            torch.cuda.synchronize()
        dist.destroy_process_group()


def ncu_traffic(sig):
    """DRAM bytes per launch of a GEMM signature from the newest committed `ncu --set full` summary that lists it
    (profiles/*_ncu_gemm_traffic.json, written by tools/ncu_summary.py from the capture of the SAME kernels); None (and the
    reason) when no capture of the shipped kernels covers it — never a number from an older kernel."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_gemm_traffic.json")))
    for f in reversed(files):
        try:
            d = json.load(open(f))
        except Exception:   # noqa: BLE001
            continue
        key = ",".join(str(int(x)) for x in sig)
        if key in d.get("signatures", {}):
            return d["signatures"][key], os.path.basename(f)
    return None, "no ncu capture of the shipped kernels lists this signature"


def run_module_api(cfgj, t, a, torch, O, timed):
    """Throughput of the drop-in module surface: model(...) -> loss on vil_prediction -> loss.backward() -> FusedAdamW.step(),
    eager Python calls, inputs resident on the device (what vilbert/task_utils.py:313-374 + train_tasks.py:545-551 do per task)."""
    import vilbert_b200
    from vilbert_b200.optim import FusedAdamW
    import torch.nn.functional as F
    model = vilbert_b200.VILBertForVLTasks(vilbert_b200.BertConfig.from_dict(cfgj), num_labels=1, precision=a.precision)
    model.train()
    groups = [{"params": [p], "lr": 1e-4 if "vil_" in n else 4e-5, "weight_decay": 0.0 if any(nd in n for nd in ("bias", "LayerNorm.bias", "LayerNorm.weight")) else 0.01}
              for n, p in model.named_parameters()]
    opt = FusedAdamW(groups, lr=4e-5, correct_bias=False, model=model)
    dev = next(model.parameters()).device
    inp = {k: v.to(dev) for k, v in t["host"][0].items()}
    tgt = t["plan"].vqa_target.clone()

    def one(i):
        out = model(inp["input_txt"], inp["input_imgs"], inp["image_loc"], inp["token_type_ids"], inp["attention_mask"], inp["image_attention_mask"])
        loss = F.binary_cross_entropy_with_logits(out[0], tgt, reduction="mean") * tgt.size(1)
        loss.backward()
        opt.step()
        model.zero_grad()

    for i in range(4):
        one(i)
    n = max(min(a.steps, 20), 5)
    ms = timed(one, n) / n
    pairs = t["B"] * t["plan"].Nv * t["plan"].Nt
    del model, opt
    torch.cuda.empty_cache()
    return {"ms_per_step": ms, "value": pairs / (ms / 1e3), "unit": "pairs/s",
            "what": "VILBertForVLTasks.forward (all 9 heads returned) + torch BCE loss + loss.backward() + FusedAdamW.step() + model.zero_grad(), train mode, device-resident inputs"}


if __name__ == "__main__":
    main()
