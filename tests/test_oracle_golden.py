"""The oracle (oracle/vilbert_oracle.py) against the fixtures that oracle/make_golden.py produced from the
UNMODIFIED reference (vilbert/vilbert.py) in the build container. Runs anywhere (CPU, no reference needed)."""
import json
import os

import pytest
import torch

from oracle import vilbert_oracle as O

CASES_FULL = ["tiny_b4", "tiny_tasktok_odd_b3", "tiny_peaked_b2"]
CASES_SUMMARY = ["base_2layer_2conect_cfg1"]


def rel(a, b):
    return ((a - b).abs().max() / (b.abs().max() + 1e-30)).item()


def _run(meta, grads):
    cfg = O.make_config(meta["config"])
    P = O.synth_params(cfg, seed=meta["seed"], qk_scale=meta["qk_scale"])
    inp = O.synth_inputs(cfg, meta["B"], meta["Nv"], meta["Nt"], seed=1234 + meta["seed"])
    Pg = {k: v.clone().requires_grad_(grads) for k, v in P.items() if k != "cls.predictions.decoder.weight"}
    Pg["cls.predictions.decoder.weight"] = Pg["bert.embeddings.word_embeddings.weight"]
    bert_o, heads_o = O.vilbert_for_vl_tasks(Pg, cfg, inp["input_txt"], inp["input_imgs"], inp["image_loc"], inp["token_type_ids"],
                                             inp["attention_mask"], inp["image_attention_mask"], inp["co_attention_mask"], inp["task_ids"])
    if grads:
        tgt = O.synth_vqa_target(meta["B"], 3129)
        l = O.vqa_loss(heads_o[0], tgt)
        for h in heads_o[1:]:
            l = l + 0.1 * h.float().clamp(-50, 50).pow(2).mean()
        l.backward()
    return inp, Pg, dict(zip(O.BERT_OUT_NAMES, bert_o)), dict(zip(O.HEAD_NAMES, heads_o))


@pytest.mark.parametrize("name", CASES_FULL)
def test_oracle_matches_reference_tensors(name, golden_dir):
    """Full tensors saved from the reference: outputs and parameter gradients (fp32, 1e-5 relative)."""
    meta = json.load(open(os.path.join(golden_dir, name + ".json")))
    gold = torch.load(os.path.join(golden_dir, name + ".pt"))
    inp, Pg, bert_o, heads_o = _run(meta, grads=True)
    for k, v in gold["inputs"].items():          # the synthetic inputs themselves are part of the contract
        assert torch.equal(inp[k], v), k
    for k, v in gold["bert"].items():
        assert rel(bert_o[k], v) < 1e-5, k
    for k, v in gold["heads"].items():
        assert rel(heads_o[k], v) < 1e-5, k
    for k, v in gold["grads"].items():
        if k.endswith(("key.bias", "key1.bias", "key2.bias")):
            # zero in exact arithmetic (the softmax over the keys ignores a shift common to all of them): both tensors hold
            # rounding noise whose bits depend on the CPU's vector width, so the difference is scaled by the key weight's gradient
            assert (Pg[k].grad - v).abs().max() <= 1e-5 * gold["grads"][k[:-4] + "weight"].abs().max(), k
            continue
        assert rel(Pg[k].grad, v) < 1e-5, k
    # q_dense1/2 never receive a gradient (vilbert.py:834,841)
    assert all(Pg[k].grad is None for k in Pg if "q_dense" in k)


@pytest.mark.parametrize("name", CASES_SUMMARY)
def test_oracle_matches_reference_summaries(name, golden_dir):
    """BASELINE.json configs[0] (bert_base_2layer_2conect forward, B=2, 36 regions, 20 tokens): sampled values and
    norms of every output recorded from the reference."""
    meta = json.load(open(os.path.join(golden_dir, name + ".json")))
    _, _, bert_o, heads_o = _run(meta, grads=False)
    outs = {**bert_o, **heads_o}
    for k, s in meta["outputs"].items():
        t = outs[k].detach().double().flatten()
        assert list(outs[k].shape) == s["shape"], k
        got = t[torch.tensor(s["sample_idx"])]
        ref = torch.tensor(s["samples"], dtype=torch.float64)
        assert (got - ref).abs().max().item() <= 1e-5 * max(s["absmax"], 1e-12), k
        assert abs(t.norm().item() - s["l2"]) <= 1e-5 * s["l2"] + 1e-12, k


def test_pretraining_losses_golden(golden_dir):
    meta = json.load(open(os.path.join(golden_dir, "tiny_pretraining_losses.json")))
    cfg = O.make_config(meta["config"])
    B, Nv, Nt = meta["B"], meta["Nv"], meta["Nt"]
    P = O.synth_params(cfg, seed=3, with_task_heads=False)
    inp = O.synth_inputs(cfg, B, Nv, Nt, seed=77)
    g = torch.Generator().manual_seed(5)
    lm = torch.full((B, Nt), -1, dtype=torch.long)
    sel = torch.rand(B, Nt, generator=g) < 0.15; sel[:, 1] = True
    lm[sel] = torch.randint(0, cfg["vocab_size"], (int(sel.sum()),), generator=g)
    il = torch.full((B, Nv - 1), -1, dtype=torch.long); il[torch.rand(B, Nv - 1, generator=g) < 0.15] = 1; il[:, 0] = 1
    it = torch.softmax(torch.randn(B, Nv - 1, cfg["v_target_size"], generator=g), -1)
    ns = torch.randint(0, 2, (B,), generator=g)
    losses = O.pretraining_losses(P, cfg, inp["input_txt"], inp["input_imgs"], inp["image_loc"], inp["token_type_ids"], inp["attention_mask"],
                                  inp["image_attention_mask"], lm, il, it, ns)
    for got, ref in zip(losses, meta["losses"]):
        assert abs(got.item() - ref) <= 1e-5 * abs(ref)


def test_param_inventory_matches_reference_names(golden_dir):
    """The oracle's parameter inventory equals the reference state_dict recorded in the fixture grads + never-grad params."""
    meta = json.load(open(os.path.join(golden_dir, "base_6layer_6conect_b4.json")))
    shapes = O.param_shapes(O.make_config(meta["config"]))
    for k, s in meta["grads"].items():
        assert list(shapes[k]) == s["shape"], k
    n = sum(int(torch.tensor(v).prod()) for k, v in shapes.items() if k != "cls.predictions.decoder.weight")
    assert abs(n / 1e6 - 268.0) < 0.1   # SURVEY.md: 268.0 M parameters for base-6-6


def test_fast_mode_golden(golden_dir):
    """config.fast_mode (text batch 1 broadcast to the image batch at the first connection layer, vilbert.py:1042-1053): sampled
    values and norms of the nine head outputs recorded from the reference (oracle/make_golden.py::check_fast_mode)."""
    meta = json.load(open(os.path.join(golden_dir, "tiny_fast_mode.json")))
    cfg = O.make_config(meta["config"])
    P = O.synth_params(cfg, seed=meta["seed"])
    inp = O.synth_inputs(cfg, meta["B"], meta["Nv"], meta["Nt"], seed=meta["input_seed"])
    with torch.no_grad():
        _, heads = O.vilbert_for_vl_tasks(P, cfg, inp["input_txt"][:1], inp["input_imgs"], inp["image_loc"], inp["token_type_ids"][:1],
                                          inp["attention_mask"][:1], inp["image_attention_mask"])
    for k, t in zip(O.HEAD_NAMES, heads):
        s = meta["outputs"][k]
        t = t.detach().double().flatten()
        assert list(heads[O.HEAD_NAMES.index(k)].shape) == s["shape"], k
        got = t[torch.tensor(s["sample_idx"])]
        assert (got - torch.tensor(s["samples"], dtype=torch.float64)).abs().max().item() <= 1e-5 * max(s["absmax"], 1e-12), k
        assert abs(t.norm().item() - s["l2"]) <= 1e-5 * s["l2"] + 1e-12, k


def test_dynamic_attention_golden(golden_dir):
    """config.dynamic_attention (vilbert.py:557-586): head outputs, the VQA loss and the gradients of the dyLinear gates recorded
    from the reference (oracle/make_golden.py::check_dynamic_attention, pinned at 0.0 difference)."""
    meta = json.load(open(os.path.join(golden_dir, "tiny_dynamic_attention.json")))
    cfg = O.make_config(meta["config"])
    P = O.synth_params(cfg, seed=meta["seed"])
    inp = O.synth_inputs(cfg, meta["B"], meta["Nv"], meta["Nt"], seed=meta["input_seed"])
    Pg = {k: v.clone().requires_grad_(True) for k, v in P.items() if k != "cls.predictions.decoder.weight"}
    Pg["cls.predictions.decoder.weight"] = Pg["bert.embeddings.word_embeddings.weight"]
    _, heads = O.vilbert_for_vl_tasks(Pg, cfg, inp["input_txt"], inp["input_imgs"], inp["image_loc"], inp["token_type_ids"],
                                      inp["attention_mask"], inp["image_attention_mask"])
    loss = O.vqa_loss(heads[0], O.synth_vqa_target(meta["B"], 3129))
    loss.backward()
    assert abs(loss.item() - meta["loss"]) <= 1e-5 * abs(meta["loss"])

    def check(t, s, k):
        t = t.detach().double().flatten()
        got = t[torch.tensor(s["sample_idx"])]
        assert (got - torch.tensor(s["samples"], dtype=torch.float64)).abs().max().item() <= 1e-5 * max(s["absmax"], 1e-12), k
        assert abs(t.norm().item() - s["l2"]) <= 1e-5 * s["l2"] + 1e-12, k
    for k, t in zip(O.HEAD_NAMES, heads):
        check(t, meta["outputs"][k], k)
    assert len(meta["gate_grads"]) == 4 * cfg["v_num_hidden_layers"]
    for k, s in meta["gate_grads"].items():
        check(Pg[k].grad, s, k)


def test_train_mode_dropout_golden(golden_dir):
    """Train mode: outputs and loss recorded from the unmodified reference whose nn.Dropout modules were replaced, by module path,
    with the engine's stateless masks (oracle/make_golden.py::check_train_mode_dropout_placement, pinned at 0.0 difference incl.
    all gradients). oracle.DropMasks must reproduce them: dropout placement, per-site probability and mask indexing."""
    meta = json.load(open(os.path.join(golden_dir, "tiny_train_mode_dropout.json")))
    cfg = O.make_config(meta["config"])
    assert len(meta["sites"]) == 35 and len(set(meta["sites"].values())) == 5
    P = O.synth_params(cfg, seed=meta["seed"])
    inp = O.synth_inputs(cfg, meta["B"], meta["Nv"], meta["Nt"], seed=meta["input_seed"])
    with torch.no_grad():
        _, heads = O.vilbert_for_vl_tasks(P, cfg, inp["input_txt"], inp["input_imgs"], inp["image_loc"], inp["token_type_ids"],
                                          inp["attention_mask"], inp["image_attention_mask"], drop=O.DropMasks(meta["step"], head_p=meta["head_p"]))
        _, heads_eval = O.vilbert_for_vl_tasks(P, cfg, inp["input_txt"], inp["input_imgs"], inp["image_loc"], inp["token_type_ids"],
                                               inp["attention_mask"], inp["image_attention_mask"])
    assert (heads[0] - heads_eval[0]).abs().max().item() > 1e-2 * heads_eval[0].abs().max().item()
    for k, t in zip(O.HEAD_NAMES, heads):
        s = meta["outputs"][k]
        t = t.detach().double().flatten()
        got = t[torch.tensor(s["sample_idx"])]
        assert (got - torch.tensor(s["samples"], dtype=torch.float64)).abs().max().item() <= 1e-5 * max(s["absmax"], 1e-12), k
        assert abs(t.norm().item() - s["l2"]) <= 1e-5 * s["l2"] + 1e-12, k


@pytest.mark.parametrize("vt", [1, 2])
def test_visual_target_golden(golden_dir, vt):
    """config.visual_target 1 / 2: the three pre-training losses recorded from the reference (for 2 with the negatives the
    reference sampled, recorded in the fixture; oracle/make_golden.py::check_visual_targets pins losses and gradients at 0.0)."""
    meta = json.load(open(os.path.join(golden_dir, f"tiny_visual_target_{vt}.json")))
    cfg = O.make_config(meta["config"])
    B, Nv, Nt = meta["B"], meta["Nv"], meta["Nt"]
    P = O.synth_params(cfg, seed=3, with_task_heads=False)
    inp = O.synth_inputs(cfg, B, Nv, Nt, seed=77)
    g = torch.Generator().manual_seed(5)
    lm = torch.full((B, Nt), -1, dtype=torch.long); lm[:, 1] = torch.randint(0, cfg["vocab_size"], (B,), generator=g)
    il = torch.full((B, Nv - 1), -1, dtype=torch.long); il[:, 0] = 1; il[:, 3] = 1; il[2, 7] = 1
    it = torch.randn(B, Nv - 1, 48, generator=g)
    ns = torch.randint(0, 2, (B,), generator=g)
    neg = torch.tensor(meta["neg_index"]) if vt == 2 else None
    with torch.no_grad():
        lo = O.pretraining_losses(P, cfg, inp["input_txt"], inp["input_imgs"], inp["image_loc"], inp["token_type_ids"], inp["attention_mask"],
                                  inp["image_attention_mask"], lm, il, it, ns, neg_index=neg)
    for a, b in zip(lo, meta["losses"]):
        assert abs(a.item() - b) <= 1e-5 * abs(b)
    if vt == 2:
        # the oracle's sampler reproduces the reference's draw order under the same seed; negatives never include the sample / region itself
        torch.manual_seed(meta["seed"])
        again = O.nce_negative_indices(B, Nv - 1, cfg["num_negative"])
        assert torch.equal(again, neg)
        R = Nv - 1
        own = torch.arange(B).view(B, 1, 1)
        assert (neg[:, :, :14] // R != own).all() and (neg[:, :, 14:] // R == own).all()
        assert (neg[:, :, 14:] % R != torch.arange(R).view(1, R, 1)).all()


def test_roberta_golden(golden_dir):
    """config.model == "roberta": the reference's RobertaEmbeddings position-id shift is overwritten inside BertEmbeddings.forward
    (vilbert.py:347-351), so the outputs recorded from the reference with model="roberta" are the ones the oracle computes with
    BERT embeddings (oracle/make_golden.py::check_roberta)."""
    meta = json.load(open(os.path.join(golden_dir, "tiny_roberta.json")))
    assert meta["config"]["model"] == "roberta" and meta["pin"]["task_tokens_run_in_reference"] is False
    cfg = O.make_config(meta["config"])
    P = O.synth_params(cfg, seed=meta["seed"])
    inp = O.synth_inputs(cfg, meta["B"], meta["Nv"], meta["Nt"], seed=meta["input_seed"])
    with torch.no_grad():
        _, heads = O.vilbert_for_vl_tasks(P, cfg, inp["input_txt"], inp["input_imgs"], inp["image_loc"], inp["token_type_ids"],
                                          inp["attention_mask"], inp["image_attention_mask"])
    for k, t in zip(O.HEAD_NAMES, heads):
        s = meta["outputs"][k]
        t = t.detach().double().flatten()
        got = t[torch.tensor(s["sample_idx"])]
        assert (got - torch.tensor(s["samples"], dtype=torch.float64)).abs().max().item() <= 1e-5 * max(s["absmax"], 1e-12), k
        assert abs(t.norm().item() - s["l2"]) <= 1e-5 * s["l2"] + 1e-12, k


def test_fixed_layers_golden(golden_dir):
    """config.fixed_t_layer: the set of parameters without a gradient and the loss recorded from the reference."""
    meta = json.load(open(os.path.join(golden_dir, "tiny_fixed_layers.json")))
    cfg = O.make_config(meta["config"])
    P = O.synth_params(cfg, seed=0)
    inp = O.synth_inputs(cfg, meta["B"], meta["Nv"], meta["Nt"], seed=1234)
    Pg = {k: v.clone().requires_grad_(True) for k, v in P.items() if k != "cls.predictions.decoder.weight"}
    Pg["cls.predictions.decoder.weight"] = Pg["bert.embeddings.word_embeddings.weight"]
    _, heads = O.vilbert_for_vl_tasks(Pg, cfg, inp["input_txt"], inp["input_imgs"], inp["image_loc"], inp["token_type_ids"], inp["attention_mask"],
                                      inp["image_attention_mask"])
    loss = O.vqa_loss(heads[0], O.synth_vqa_target(meta["B"], 3129))
    loss.backward()
    assert abs(loss.item() - meta["loss"]) <= 1e-5 * abs(meta["loss"])
    frozen = sorted(k for k, v in Pg.items() if k != "cls.predictions.decoder.weight" and (v.grad is None or v.grad.abs().max() == 0))
    assert frozen == meta["frozen"]


def test_in_batch_pairs_golden(golden_dir):
    """config.in_batch_pairs: BertModel outputs at batch b^2 recorded from the reference."""
    meta = json.load(open(os.path.join(golden_dir, "tiny_in_batch_pairs.json")))
    cfg = O.make_config(meta["config"])
    P = O.synth_params(cfg, seed=meta["seed"])
    inp = O.synth_inputs(cfg, meta["B"], meta["Nv"], meta["Nt"], seed=meta["input_seed"])
    with torch.no_grad():
        outs = O.bert_model(P, cfg, inp["input_txt"], inp["input_imgs"], inp["image_loc"], inp["token_type_ids"], inp["attention_mask"], inp["image_attention_mask"])
    for k, t in zip(O.BERT_OUT_NAMES, outs):
        s = meta["outputs"][k]
        assert list(t.shape) == s["shape"] and t.shape[0] == meta["B"] ** 2, k
        t = t.detach().double().flatten()
        assert (t[torch.tensor(s["sample_idx"])] - torch.tensor(s["samples"], dtype=torch.float64)).abs().max().item() <= 1e-5 * max(s["absmax"], 1e-12), k
        assert abs(t.norm().item() - s["l2"]) <= 1e-5 * s["l2"] + 1e-12, k


def test_visualization_golden(golden_dir):
    """config.visualization: attention probabilities of the last text layer and last connection layer recorded from the reference."""
    meta = json.load(open(os.path.join(golden_dir, "tiny_visualization.json")))
    cfg = O.make_config(meta["config"])
    P = O.synth_params(cfg, seed=meta["seed"])
    inp = O.synth_inputs(cfg, meta["B"], meta["Nv"], meta["Nt"], seed=meta["input_seed"])
    got = {}
    O.ATTN_HOOK = lambda name, p, q, k: got.__setitem__(name, p)
    try:
        with torch.no_grad():
            O.vilbert_for_vl_tasks(P, cfg, inp["input_txt"], inp["input_imgs"], inp["image_loc"], inp["token_type_ids"], inp["attention_mask"], inp["image_attention_mask"])
    finally:
        O.ATTN_HOOK = None
    nl, nc = cfg["num_hidden_layers"] - 1, len(cfg["v_biattention_id"]) - 1
    for key, name in (("attn_text_last", f"bert.encoder.layer.{nl}.attention.self.dropout"), ("attn1_last", f"bert.encoder.c_layer.{nc}.biattention.dropout1"),
                      ("attn2_last", f"bert.encoder.c_layer.{nc}.biattention.dropout2")):
        s, t = meta[key], got[name]
        assert list(t.shape) == s["shape"], key
        t = t.double().flatten()
        assert (t[torch.tensor(s["sample_idx"])] - torch.tensor(s["samples"], dtype=torch.float64)).abs().max().item() <= 1e-5 * max(s["absmax"], 1e-12), key
