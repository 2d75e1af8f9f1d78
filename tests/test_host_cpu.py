"""CPU-side checks of the host code: C-ABI exports, config semantics, parameter layout, plan construction."""
import ctypes
import json
import os

import pytest
import torch

from oracle import vilbert_oracle as O
from vilbert_b200 import _lib as L
from vilbert_b200.config import BertConfig
from vilbert_b200.engine import Engine, ParamStore


def test_library_exports_every_declared_symbol():
    lib = L.lib()
    declared = L.exported_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/vilbert_b200.h but not exported"
    assert set(L._SIGNATURES) <= set(declared)
    assert lib.vb_version() == 2
    assert ctypes.sizeof(L.GemmArgs) >= 160 and ctypes.sizeof(L.AttnArgs) >= 150


_NO_GPU_CHILD = r"""
import json, os, sys
sys.path.insert(0, sys.argv[1])
import torch
assert not torch.cuda.is_available()
from vilbert_b200 import _lib as L, modeling
from vilbert_b200.config import BertConfig
from vilbert_b200.engine import Engine
cfg = BertConfig.from_dict(json.load(open(os.path.join(sys.argv[1], "tests", "golden", "tiny_b4.json")))["config"])
for name, make in (("VILBertForVLTasks", lambda: modeling.VILBertForVLTasks(cfg, num_labels=1)), ("Engine", lambda: Engine(cfg, "cpu"))):
    try:
        make()
    except L.VBError:
        continue
    raise SystemExit(name + " did not raise VBError")
"""


def test_no_fallback_without_gpu():
    """The product must fail loudly when it cannot run on the GPU: no CPU path. Checked in a child process that sees no CUDA
    device, so that it runs on GPU machines too."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _NO_GPU_CHILD, root], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]


def test_config_semantics(tmp_path, golden_dir):
    cfgj = json.load(open(os.path.join(golden_dir, "base_6layer_6conect_b4.json")))["config"]
    p = tmp_path / "c.json"
    p.write_text(json.dumps(cfgj))
    c = BertConfig.from_json_file(str(p))
    assert c.hidden_size == 768 and c.v_hidden_size == 1024 and c.bi_num_attention_heads == 8
    assert c.v_biattention_id == [0, 1, 2, 3, 4, 5] and c.t_biattention_id == [6, 7, 8, 9, 10, 11]
    # defaults the JSON does not carry (vilbert.py:158-184) and post-hoc mutation
    assert c.fusion_method == "mul" and c.task_specific_tokens is False and c.with_coattention is True
    c.task_specific_tokens = True
    assert json.loads(c.to_json_string())["task_specific_tokens"] is True
    c2 = BertConfig(30522, hidden_size=768)
    assert c2.vocab_size == 30522 and c2.v_feature_size == 2048
    with pytest.raises(ValueError):
        BertConfig(3.5)
    BertConfig.from_dict(dict(cfgj, dynamic_attention=True)).check_supported()
    for bad in (dict(cfgj, dynamic_attention=True, in_batch_pairs=True), dict(cfgj, hidden_act="relu")):
        with pytest.raises(NotImplementedError):
            BertConfig.from_dict(bad).check_supported()
    BertConfig.from_dict(dict(cfgj, model="roberta")).check_supported()      # same embeddings as BERT in the reference (tiny_roberta.json)
    with pytest.raises(NotImplementedError):
        BertConfig.from_dict(dict(cfgj, model="roberta", task_specific_tokens=True)).check_supported()


def test_param_store_layout(golden_dir):
    cfgj = json.load(open(os.path.join(golden_dir, "base_6layer_6conect_b4.json")))["config"]
    cfg = BertConfig.from_dict(cfgj)
    ps = ParamStore(cfg, "cpu")
    ref = O.param_shapes(O.make_config(cfgj))
    ref.pop("cls.predictions.decoder.weight")
    assert {k: tuple(v[1]) for k, v in ps.entries.items()} == {k: tuple(v) for k, v in ref.items()}
    # fused QKV views alias the three reference tensors, in order
    p = "bert.encoder.layer.3.attention.self"
    ps.p(p + ".query.weight").fill_(1.0); ps.p(p + ".key.weight").fill_(2.0); ps.p(p + ".value.weight").fill_(3.0)
    w = ps.p(p + ".qkv.weight")
    assert w.shape == (3 * 768, 768)
    assert w[:768].eq(1).all() and w[768:1536].eq(2).all() and w[1536:].eq(3).all()
    for name, (off, shape) in list(ps.entries.items()) + list(ps.fused.items()):
        assert off % 8 == 0, name     # 16-byte aligned bf16 shadow / 32-byte aligned fp32
    assert ps.p("bert.encoder.c_layer.0.biattention.qkv2.weight").shape == (3 * 1024, 768)


@pytest.mark.parametrize("task_tokens,B", [(False, 4), (True, 3)])
def test_plan_builds_on_cpu(golden_dir, task_tokens, B):
    """Plans are pure host data (buffers + C-ABI call records): build them here without a GPU and check structure."""
    cfgj = dict(json.load(open(os.path.join(golden_dir, "tiny_b4.json")))["config"], task_specific_tokens=task_tokens)
    eng = Engine(BertConfig.from_dict(cfgj), "cpu", _build_only=True)
    fwd_only = eng.plan(B, 9, 11)
    assert fwd_only.n_kernels_bwd == 0 and fwd_only.n_kernels_fwd > 50
    full = eng.plan(B, 9, 11, grad_outputs=O.HEAD_NAMES)
    vqa = eng.plan(B, 9, 11, grad_outputs=("vil_prediction",), vqa_loss=True)
    assert full.n_kernels_fwd == fwd_only.n_kernels_fwd == vqa.n_kernels_fwd
    assert full.n_kernels_bwd > vqa.n_kernels_bwd > full.n_kernels_fwd      # dead head branches are not emitted
    assert set(O.HEAD_NAMES) | set(O.BERT_OUT_NAMES) == set(full.outputs)
    nt = 9 + int(task_tokens)
    assert tuple(full.outputs["sequence_output_t"].shape) == (B, nt, cfgj["hidden_size"])
    assert tuple(full.outputs["linguisic_prediction"].shape) == (B, nt, cfgj["vocab_size"])
    assert tuple(full.outputs["vil_binary_prediction"].shape) == ((B // 2, 2) if B % 2 == 0 else (B, 2))
    bert_only = eng.plan(B, 9, 11, heads="none")
    assert set(bert_only.outputs) == set(O.BERT_OUT_NAMES)


def _op_names(ops):
    return [getattr(op[0], "__name__", None) or getattr(op[0], "_name", "") for op in ops if op[0] is not None]


def test_special_mode_plans_build_on_cpu(golden_dir):
    """Structure of the plans of the optional modes, checked without a GPU: dynamic_attention (gate parameters, pooling / gate ops
    in both passes, data-parallel pieces still tile the gradient buffer) and the compacted masked-LM head of the fused pre-training
    objective (no [tokens, vocab] logits output, capacity arithmetic, cache key)."""
    from vilbert_b200.engine import LOSS_HEADS
    tiny = json.load(open(os.path.join(golden_dir, "tiny_b4.json")))["config"]
    cfgj = dict(tiny, dynamic_attention=True)
    eng = Engine(BertConfig.from_dict(cfgj), "cpu", _build_only=True)
    names = set(eng.ps.entries)
    assert names == set(O.param_shapes(O.make_config(cfgj))) - {"cls.predictions.decoder.weight"} | {"bert.embeddings.word_embeddings.weight"}
    p0 = "bert.encoder.v_layer.0.attention.self"
    (wq, sq), (wk, sk) = eng.ps.entries[p0 + ".dyLinear_q.weight"], eng.ps.entries[p0 + ".dyLinear_k.weight"]
    assert sq == sk == (cfgj["v_hidden_size"], cfgj["hidden_size"]) and wk == wq + sq[0] * sq[1]       # contiguous: one fused [2Hv, Ht] GEMM
    assert eng.ps.fused[p0 + ".dy.weight"] == (wq, (2 * sq[0], sq[1]))
    plan = eng.plan(4, 9, 11, grad_outputs=O.HEAD_NAMES, train=True)
    base = Engine(BertConfig.from_dict(tiny), "cpu", _build_only=True).plan(4, 9, 11, grad_outputs=O.HEAD_NAMES, train=True)
    nv = cfgj["v_num_hidden_layers"]
    f, b = _op_names(plan.fwd), _op_names(plan.bwd)
    assert f.count("vb_gate_scale_fwd") == nv and b.count("vb_gate_scale_bwd") == nv
    assert 1 <= f.count("vb_masked_mean_fwd") <= nv and b.count("vb_masked_mean_bwd") == f.count("vb_masked_mean_fwd")
    assert plan.n_kernels_fwd > base.n_kernels_fwd and plan.n_kernels_bwd > base.n_kernels_bwd
    segs = plan.ddp_segments(4)
    assert segs[0][3] == eng.ps.numel and segs[-1][2] == 0 and all(nx[3] == cur[2] for cur, nx in zip(segs, segs[1:]))
    for (lo, hi, glo, ghi) in segs:
        for (off, n), touch in plan.grad_touch.items():
            if glo <= off < ghi:
                assert touch < hi
    # compacted masked-LM head
    engp = Engine(BertConfig.from_dict(tiny), "cpu", heads="pretraining", _build_only=True)
    B, Nt = 64, 20
    pc = engp.plan(B, Nt, 11, grad_outputs=LOSS_HEADS["pretraining"], loss="pretraining")
    assert "linguisic_prediction" not in pc.outputs and pc.lm_c["cap"] == 320 and tuple(pc.lm_c["logits"].shape) == (320, tiny["vocab_size"])
    assert set(pc.loss_inputs) == {"masked_lm_labels", "image_target", "image_label", "next_sentence_label"}
    assert (pc.loss_inputs["masked_lm_labels"] == -1).all()                     # nothing labelled until the caller loads labels
    engp.lm_capacity = 0.5
    assert engp.plan(B, Nt, 11, grad_outputs=LOSS_HEADS["pretraining"], loss="pretraining").lm_c["cap"] == 640
    engp.lm_compact = False
    pf = engp.plan(B, Nt, 11, grad_outputs=LOSS_HEADS["pretraining"], loss="pretraining")
    assert pf.lm_c is None and tuple(pf.outputs["linguisic_prediction"].shape) == (B, Nt, tiny["vocab_size"])
    assert pf is not pc and len(engp.plans) == 3
    small = Engine(BertConfig.from_dict(tiny), "cpu", heads="pretraining", _build_only=True).plan(4, 9, 11, grad_outputs=LOSS_HEADS["pretraining"], loss="pretraining")
    assert small.lm_c["cap"] == 40                                              # never more rows than there are (8-padded)


def test_shared_activation_arena_layout(golden_dir):
    """Engine.enable_activation_arena: activation / scratch buffers of every plan are sub-allocated from one arena (plans overlay
    each other), while everything loaded or initialised outside a run (inputs, targets, output gradients) stays private."""
    from vilbert_b200._lib import VBError
    cfgj = json.load(open(os.path.join(golden_dir, "tiny_b4.json")))["config"]
    plain = Engine(BertConfig.from_dict(cfgj), "cpu", _build_only=True).plan(4, 9, 11, grad_outputs=("vil_prediction",), vqa_loss=True)
    eng = Engine(BertConfig.from_dict(cfgj), "cpu", _build_only=True)
    eng.enable_activation_arena(64 << 20)
    a = eng.plan(4, 9, 11, grad_outputs=("vil_prediction",), vqa_loss=True)
    b = eng.plan(6, 20, 33, grad_outputs=("vil_prediction",), vqa_loss=True)
    assert (a.n_kernels_fwd, a.n_kernels_bwd) == (plain.n_kernels_fwd, plain.n_kernels_bwd)
    lo, hi = eng.arena.data_ptr(), eng.arena.data_ptr() + eng.arena.numel()
    inside = lambda t: lo <= t.data_ptr() < hi
    for p in (a, b):
        assert not any(inside(t) for t in (p.in_ids, p.in_tt, p.in_amask, p.in_imask, p.in_feat, p.in_loc, p.vqa_target, p.loss))
        assert all(inside(t) for t in (p.outputs["sequence_output_t"], p.outputs["vil_prediction"], p.mask_t, p.mask_v))
        assert 0 < p.arena_bytes <= eng.arena.numel() and p.arena_bytes % 256 == 0
    assert a.mask_t.data_ptr() == b.mask_t.data_ptr() and b.arena_bytes > a.arena_bytes       # same offsets: the plans overlay
    private = lambda p: sum(t.numel() * t.element_size() for t in p._keep if torch.is_tensor(t))
    assert private(a) < 0.1 * private(plain)
    with pytest.raises(VBError):
        eng.enable_activation_arena(1 << 20)          # only before the first plan
    small = Engine(BertConfig.from_dict(cfgj), "cpu", _build_only=True)
    small.enable_activation_arena(1 << 20)
    with pytest.raises(VBError):
        small.plan(4, 9, 11)


def test_ddp_segments_partition_the_gradient_buffer(golden_dir):
    """Overlapped data-parallel step: backward pieces (each with at least one kernel, no side-stream event recorded in one
    piece and waited for in a later one) release tail ranges of the flat gradient buffer that (a) tile it exactly and (b)
    are never written by a later backward op."""
    cfgj = json.load(open(os.path.join(golden_dir, "tiny_b4.json")))["config"]
    eng = Engine(BertConfig.from_dict(cfgj), "cpu", _build_only=True)
    plan = eng.plan(4, 9, 11, grad_outputs=O.HEAD_NAMES, train=True)
    for k in (1, 3, 8):
        segs = plan.ddp_segments(k)
        assert segs[0][0] == 0 and segs[-1][1] == len(plan.bwd) and segs[0][3] == eng.ps.numel and segs[-1][2] == 0
        for (lo, hi, glo, ghi), nxt in zip(segs, segs[1:] + [None]):
            assert lo < hi and glo <= ghi
            assert any(op[0] is not None for op in plan.bwd[lo:hi])                          # no kernel-less piece
            recs = {op[1][1] for op in plan.bwd[:hi] if op[0] is None and len(op[1]) == 2 and op[1][0] == "rec"}
            late = {op[1][1] for op in plan.bwd[hi:] if op[0] is None and len(op[1]) == 2 and op[1][0] == "wait"}
            assert not (recs & late)                                                          # no event crosses the cut
            if nxt is not None:
                assert nxt[0] == hi and nxt[3] == glo
            for (off, n), touch in plan.grad_touch.items():                              # released ranges are final
                if off >= glo and off < ghi:
                    assert touch < hi, (off, touch, hi)
    # execution-order layout: the tied word-embedding table (written first AND last in backward) sits at offset 0
    assert eng.ps.entries["bert.embeddings.word_embeddings.weight"][0] == 0


def test_gemm_tile_configuration_cost_model():
    """vb_gemm_plan (host only): the (tile width, CTA pairing, k splits) vb_gemm_bf16 picks for the model's GEMM shapes on a
    148-SM device — CTA pairs with 256-wide tiles for the large image-stream problems, single-CTA 128-wide tiles where the tile
    count binds, split-K only for the weight-gradient form; caller-fixed values are honoured, nonsense is rejected."""
    import ctypes as C
    from vilbert_b200 import _lib as L
    lib = L.lib()

    def plan(M, N, K, sms=148, **kw):
        g = L.GemmArgs(); g.M, g.N, g.K, g.alpha = M, N, K, 1.0
        g.A = g.B = 0x1000                                     # never dereferenced by the query
        g.block_n, g.cluster_m = kw.get("block_n", 0), kw.get("cluster_m", 0)
        if kw.get("atomic"):
            g.atomic_out, g.out_f32, g.split_k = 1, 0x1000, kw.get("split_k", 0)
        else:
            g.split_k = kw.get("split_k", 1)
            if kw.get("bf16"): g.out_bf16 = 0x1000
            else: g.out_f32 = 0x1000
            if kw.get("res"): g.residual = 0x1000
        bn, cl, sp = C.c_int32(), C.c_int32(), C.c_int32()
        st = lib.vb_gemm_plan(C.byref(g), sms, C.byref(bn), C.byref(cl), C.byref(sp))
        return st, (bn.value, cl.value, sp.value)

    assert plan(6400, 3072, 1024, bf16=True) == (0, (256, 2, 1))          # image QKV: 256 x 256 pair tiles
    assert plan(8192, 8192, 8192, bf16=True) == (0, (256, 2, 1))
    assert plan(2304, 768, 768, res=True) == (0, (128, 1, 1))             # text out-proj: 108 tiles on 148 SMs
    st, (bn, cl, sp) = plan(3072, 1024, 6400, atomic=True)                # image QKV weight gradient
    assert st == 0 and (bn, cl) == (256, 2) and sp > 1
    st, (bn, cl, sp) = plan(768, 768, 2304, atomic=True)
    assert st == 0 and sp > 1                                             # 36 tiles: split K to fill the SMs
    assert plan(6400, 1024, 1024, res=True)[1][2] == 1                    # no split-K outside the atomic form
    assert plan(6400, 3072, 1024, bf16=True, block_n=128, cluster_m=1) == (0, (128, 1, 1))
    assert plan(3072, 1024, 6400, atomic=True, split_k=5)[1][2] == 5
    assert plan(64, 1024, 768)[1][1] == 1                                 # one row block: nothing to pair
    assert plan(6400, 1024, 1024, block_n=64)[0] == 1 and b"block_n" in lib.vb_last_error()
    assert plan(6400, 1024, 1024, cluster_m=3)[0] == 1 and b"cluster_m" in lib.vb_last_error()
    assert plan(6400, 1024, 1024, res=True, split_k=2)[0] == 1 and b"split_k" in lib.vb_last_error()


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm beside the GPU arm): rank 0 prints ONE JSON line with the contract keys for the
    same metric / workload, other ranks print nothing and exit 0. Runs the oracle port on a 1-sample step, exactly --steps times."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", "--cpu-batch", "1"]
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == ""
    env = dict(os.environ, RANK="0", WORLD_SIZE="2", LOCAL_RANK="0")
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["unit"] == "pairs/s" and d["higher_is_better"] is True
    assert "bert_base_6layer_6conect" in d["metric"] and "bert_base_6layer_6conect" in d["config"]["workload"]
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1 and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == "port"
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}

