"""-m gpu tests of the drop-in trainer layer: compute_loss (autograd bridge) == fused engine path,
frozen-reference log-prob pre-pass vs oracle, train()/checkpoint/resume on a synthetic dataset."""
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import llava_dpo_oracle as O

pytestmark = pytest.mark.gpu


def dims():
    from rlaifv_b200.model import LlavaDims
    c = O.TINY
    return LlavaDims(vocab_size=c.vocab_size, hidden_size=c.hidden_size, intermediate_size=c.intermediate_size,
                     num_layers=c.num_layers, num_heads=c.num_heads, clip_hidden=c.clip_hidden,
                     clip_intermediate=c.clip_intermediate, clip_layers=c.clip_layers, clip_heads=c.clip_heads,
                     image_size=c.image_size, patch_size=c.patch_size)


def instances(B, seed, ragged=True):
    """(rej_dict, win_dict) tuples like DPODataset.__getitem__ yields."""
    b = O.synthetic_pair_batch(O.TINY, B, 20, 16, seed=seed, image_pos=5, ragged=ragged)
    ids, labs = b["concatenated_input_ids"], b["concatenated_labels"]
    out = []
    for i in range(B):
        def one(row, kind):
            n = int((ids[row] != 0).sum())
            return {"input_ids": ids[row, :n].clone(), "labels": labs[row, :n].clone(), "image": b["images"][i],
                    f"ref_{kind}_logp": -40.0 - i, f"ref_{kind}_avg_logp": -2.5, f"ref_{kind}_per_token_logp": [0.0] * (n + 600)}
        out.append((one(B + i, "rej"), one(i, "win")))
    return out


class Tok:
    pad_token_id = 0


def make_args(tmp, **kw):
    a = SimpleNamespace(learning_rate=1e-3, weight_decay=0.01, max_steps=4, warmup_ratio=0.0, dpo_use_average=False,
                        dpo_token_weighted=False, task="DPO", output_dir=str(tmp), logging_steps=1, save_strategy="steps",
                        save_steps=2, save_total_limit=5, per_device_train_batch_size=2, dataloader_num_workers=0,
                        lr_scheduler_type="constant", bf16=True, deepspeed=None, seed=1)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_compute_loss_autograd_bridge_equals_engine(tmp_path):
    from rlaifv_b200.collator import DataCollatorForDPODataset
    from rlaifv_b200.llava_model import LlavaLlamaForCausalLM
    from rlaifv_b200.trainers import LLaVA15DPOTrainer
    params = O.make_params(O.TINY, seed=0, scale=0.4)
    model = LlavaLlamaForCausalLM(dims(), "cuda", hf_state=params)
    coll = DataCollatorForDPODataset(tokenizer=Tok(), beta=0.1, mod_token_weight=1.0)
    trainer = LLaVA15DPOTrainer(model=model, tokenizer=Tok(), args=make_args(tmp_path), train_dataset=None,
                                data_collator=coll)
    batch = coll(instances(2, seed=3))
    loss = trainer.compute_loss(model, dict(batch))
    loss.backward()
    g_bridge = model.policy.store.grad.clone()
    m = trainer.engine.train_step(dict(batch), optimizer_step=False)
    g_engine = model.policy.store.grad.clone()
    torch.cuda.synchronize()
    assert abs(float(loss) - float(m[0])) <= 1e-5 * max(1.0, abs(float(loss)))
    assert torch.equal(g_bridge, g_engine)        # same kernels, same order -> bit-identical gradients
    logged = trainer.state["log_history"][-1]
    assert set(k for k in logged if "/" in k) == {"rewards_train/chosen", "rewards_train/rejected",
                                                  "rewards_train/accuracies", "rewards_train/margins",
                                                  "logps_train/rejected", "logps_train/chosen",
                                                  "logps_train/ref_rejected", "logps_train/ref_chosen"}


def test_reference_logp_prepass_matches_oracle():
    from rlaifv_b200.collator import preference_collator_fn
    from rlaifv_b200.data import get_multimodal_sample_logps
    from rlaifv_b200.llava_model import LlavaLlamaForCausalLM
    params = O.make_params(O.TINY, seed=0, scale=0.4)
    model = LlavaLlamaForCausalLM(dims(), "cuda", hf_state=params)
    inst = instances(3, seed=8)
    batches = [preference_collator_fn(inst[:2], 0), preference_collator_fn(inst[2:], 0)]
    outs = get_multimodal_sample_logps(model, batches)
    pb = {k: v.to(torch.bfloat16) for k, v in params.items()}
    P = O.TINY.num_patches
    for i, (rej, win) in enumerate(inst):
        for kind, d, base in (("win", win, 0), ("rej", rej, 3)):
            ids, labs = d["input_ids"][None], d["labels"][None]
            o = O.policy_logps(pb, O.TINY, torch.cat([ids, ids]), torch.cat([labs, labs]), d["image"][None].to(torch.bfloat16))
            per_tok = outs[base + 2][i]
            assert len(per_tok) == ids.shape[1] - 1 + P - 1          # T_i - 1 entries, like the reference's batch-1 pass
            ref_sum = float(o["logp"][0])
            assert abs(outs[base][i] - ref_sum) <= 1e-3 * abs(ref_sum)
            assert abs(outs[base + 1][i] - float(o["avg_logp"][0])) <= 1e-3 * abs(float(o["avg_logp"][0]))
            mask = o["labels"][0, 1:] != -100
            got = torch.tensor(per_tok)[mask]
            want = o["per_token_logps"][0][mask]
            assert float((got - want).abs().max()) <= 1e-2 * float(want.abs().max())


def test_train_loop_checkpoint_resume(tmp_path):
    from rlaifv_b200.collator import DataCollatorForDPODataset
    from rlaifv_b200.llava_model import LlavaLlamaForCausalLM
    from rlaifv_b200.trainers import LLaVA15DPOTrainer
    params = O.make_params(O.TINY, seed=0, scale=0.4)
    data = instances(8, seed=11)
    coll = DataCollatorForDPODataset(tokenizer=Tok(), beta=0.1, mod_token_weight=1.0)

    def run(max_steps, resume):
        model = LlavaLlamaForCausalLM(dims(), "cuda", hf_state=params)
        tr = LLaVA15DPOTrainer(model=model, tokenizer=Tok(), args=make_args(tmp_path, max_steps=max_steps),
                               train_dataset=data, data_collator=coll)
        tr.train(resume_from_checkpoint=resume)
        torch.cuda.synchronize()
        return model, tr

    m1, t1 = run(2, False)                       # writes checkpoint-2
    assert os.path.isdir(tmp_path / "checkpoint-2")
    m2, t2 = run(4, True)                        # resumes at step 2, runs to 4
    assert t2.state["global_step"] == 4
    losses = [h["loss"] for h in t2.state["log_history"] if "loss" in h]
    assert len(losses) == 4 and all(l == l for l in losses)      # steps 1,2 restored from the log + 3,4 new
    w0 = params["model.layers.0.mlp.down_proj.weight"].to(torch.bfloat16)
    w2 = m2.state_dict()["model.layers.0.mlp.down_proj.weight"].cpu()
    assert float((w2.float() - w0.float()).abs().max()) > 0     # parameters moved
    t2.save_state()
    assert os.path.exists(tmp_path / "trainer_state.json")


def test_train_llava15_entry_end_to_end(tmp_path, monkeypatch):
    """The shipped entry point (script/train/llava15_train.sh -> rlaifv_b200.train_llava15.train) on a tiny checkpoint:
    config.json-driven dimensions, CLIP image processor built from the vision tower's preprocessor_config.json
    (muffin/train/train_llava15.py:244), reference-log-prob pre-pass, dataset, collator, two optimisation steps."""
    import io
    import json
    from PIL import Image
    from oracle.toy_tokenizer import ToyTokenizer
    from rlaifv_b200 import data as D
    from rlaifv_b200 import train_llava15 as TL
    c = O.TINY
    params = O.make_params(c, seed=0, scale=0.4)
    ckpt, vt = tmp_path / "ckpt", tmp_path / "clip"
    ckpt.mkdir()
    vt.mkdir()
    vp = "model.vision_tower.vision_tower."
    torch.save({k: v for k, v in params.items() if not k.startswith(vp)}, ckpt / "pytorch_model.bin")
    torch.save({k[len(vp):]: v for k, v in params.items() if k.startswith(vp)}, vt / "pytorch_model.bin")
    (ckpt / "config.json").write_text(json.dumps({
        "vocab_size": c.vocab_size, "hidden_size": c.hidden_size, "intermediate_size": c.intermediate_size,
        "num_hidden_layers": c.num_layers, "num_attention_heads": c.num_heads, "rms_norm_eps": c.rms_eps}))
    (vt / "config.json").write_text(json.dumps({"vision_config": {
        "hidden_size": c.clip_hidden, "intermediate_size": c.clip_intermediate, "num_hidden_layers": c.clip_layers,
        "num_attention_heads": c.clip_heads, "image_size": c.image_size, "patch_size": c.patch_size}}))
    (vt / "preprocessor_config.json").write_text(json.dumps({
        "size": {"shortest_edge": c.image_size}, "crop_size": {"height": c.image_size, "width": c.image_size},
        "image_mean": [0.48145466, 0.4578275, 0.40821073], "image_std": [0.26862954, 0.26130258, 0.27577711]}))
    monkeypatch.setattr(D, "load_tokenizer", lambda path, max_len: ToyTokenizer())
    g = torch.Generator().manual_seed(1)
    words = "a red bus on the street near two small dogs and one cat under blue sky with trees".split()
    rows = []
    for i in range(6):
        arr = (torch.rand(70 + 10 * i, 90, 3, generator=g) * 255).to(torch.uint8).numpy()      # non-square: resize + crop
        buf = io.BytesIO()
        Image.fromarray(arr).save(buf, format="PNG")
        rows.append({"image": {"bytes": buf.getvalue()}, "question": "what is shown in picture %d ?" % i,
                     "chosen": " ".join(words[i:i + 6]), "rejected": " ".join(words[::-1][i:i + 4]), "idx": i,
                     "origin_dataset": "synthetic", "origin_split": "train", "image_path": "img%d" % i})
    out_dir = tmp_path / "out"
    tr = TL.train(argv=["--model_name_or_path", str(ckpt), "--vision_tower", str(vt), "--mm_vision_select_layer", "-2",
                        "--data_dir", str(tmp_path / "data"), "--data_source_names", "", "--data_source_weights", "1",
                        "--task", "DPO", "--dpo_beta", "0.1", "--dpo_token_weight", "1.0", "--learning_rate", "1e-3",
                        "--max_steps", "2", "--per_device_train_batch_size", "3", "--logging_steps", "1",
                        "--save_strategy", "no", "--lr_scheduler_type", "constant", "--model_max_length", "2048",
                        "--output_dir", str(out_dir), "--bf16", "True", "--image_aspect_ratio", "pad"], source_rows=rows)
    torch.cuda.synchronize()
    assert sorted(os.listdir(tmp_path / "data")) == ["RLAIF-V-Dataset-withlogp_000-6.parquet"]
    losses = [h["loss"] for h in tr.state["log_history"] if "loss" in h]
    assert len(losses) == 2 and abs(losses[0] - 0.693147) < 5e-3 and all(l == l for l in losses)
    assert all(h.get("learning_rate") == 1e-3 for h in tr.state["log_history"] if "loss" in h)
    assert os.path.exists(out_dir / "pytorch_model.bin") and os.path.exists(out_dir / "trainer_state.json")
    rej, win = tr.train_dataset[0]
    assert tuple(win["image"].shape) == (3, c.image_size, c.image_size) and win["image"].dtype == torch.float32


SEAM_FIXTURE = os.path.join(os.path.dirname(__file__), "golden", "trainer", "compute_loss_seam.npz")


def test_reference_compute_loss_text_on_rebound_seam():
    """INTEGRATION.md §1, the two-line rebinding: the reference's OWN `LLaVA15DPOTrainer.compute_loss`
    (muffin/train/trainers.py:279-311) with only `get_beta_and_logps` and `dpo_loss` rebound to this repo's, on the
    collator output below. oracle/gen_golden_trainer_seam.py ran it on a B200 and stored its loss, the metrics it logs
    and the gradient its `loss.backward()` drove through the hand-written backward (norm and a seeded sample). The
    fused engine on the same batch must give the same loss, metrics and gradients."""
    from rlaifv_b200.collator import DataCollatorForDPODataset
    from rlaifv_b200.engine import DPOStepEngine
    from rlaifv_b200.llava_model import LlavaLlamaForCausalLM
    fx = np.load(SEAM_FIXTURE)
    params = O.make_params(O.TINY, seed=0, scale=0.4)
    assert abs(O.params_checksum(params) - float(fx["params_checksum"])) <= 1e-9 * float(fx["params_checksum"])
    batch = DataCollatorForDPODataset(tokenizer=Tok(), beta=0.1, mod_token_weight=1.0)(instances(2, seed=3))
    assert np.array_equal(batch["concatenated_input_ids"].numpy(), fx["concatenated_input_ids"])
    assert np.array_equal(batch["concatenated_labels"].numpy(), fx["concatenated_labels"])
    g_bridge = torch.from_numpy(fx["grad_sample"])
    assert float(g_bridge.abs().max()) > 0
    # the fused engine on the same batch (no optimizer step): same loss, same metrics, same gradients
    model2 = LlavaLlamaForCausalLM(dims(), "cuda", hf_state=params)
    eng = DPOStepEngine(model2.policy, lr=1e-3, total_steps=4, constant_lr=True)
    m = eng.train_step(dict(batch), optimizer_step=False)
    md = eng.metrics_dict(m)
    torch.cuda.synchronize()
    assert abs(float(fx["loss"]) - md["loss"]) <= 1e-6 * max(1.0, abs(md["loss"]))
    for k in ("rewards_train/chosen", "rewards_train/rejected", "rewards_train/accuracies", "rewards_train/margins",
              "logps_train/chosen", "logps_train/rejected", "logps_train/ref_chosen", "logps_train/ref_rejected"):
        assert abs(float(fx["metric:" + k]) - md[k]) <= 1e-5 * max(1.0, abs(md[k])), k
    g_engine = model2.policy.store.grad.float()
    sample = g_engine[torch.from_numpy(fx["grad_index"]).long().cuda()].cpu()
    assert float((g_bridge - sample).norm() / sample.norm()) <= 1e-3
    assert abs(float(fx["grad_norm"]) - float(g_engine.double().norm())) <= 1e-3 * float(g_engine.double().norm())


def test_llava_token_weighted_extension_matches_spliced_oracle():
    """--dpo_token_weighted on the LLaVA policy (an EXTENSION: the reference raises NotImplementedError for it,
    trainers.py:246-248, because its collator's weights are in text positions and the per-token log-probs in spliced
    positions). The engine maps the collator's weights through the splice and applies compute_weighted_logp
    (trainers.py:128-137) to policy AND cached reference per-token log-probs in spliced positions; checked against the
    same arithmetic done with the oracle's tensors, and against the unweighted path when every weight is 1."""
    from rlaifv_b200.collator import DataCollatorForDPODataset
    from rlaifv_b200.engine import DPOStepEngine
    from rlaifv_b200.llava_model import LlavaLlamaForCausalLM
    c = O.TINY
    params = O.make_params(c, seed=0, scale=0.4)
    B = 2
    inst = instances(B, seed=7)
    # make the pair share most tokens, so the diff-based weights are non-trivial (3.0 on modified spans)
    for rej, win in inst:
        n = min(len(rej["input_ids"]), len(win["input_ids"]))
        rej["input_ids"][6:n - 6] = win["input_ids"][6:n - 6]
        rej["labels"] = torch.where(rej["labels"] != -100, rej["input_ids"], rej["labels"])
    # cached reference per-token log-probs in SPLICED positions, as the pre-pass stores them
    g = torch.Generator().manual_seed(3)
    for rej, win in inst:
        for d, kind in ((rej, "rej"), (win, "win")):
            n_sp = len(d["input_ids"]) - 1 + c.num_patches
            d[f"ref_{kind}_per_token_logp"] = (-2.0 + 0.5 * torch.randn(n_sp - 1, generator=g)).tolist()
    coll = DataCollatorForDPODataset(tokenizer=Tok(), beta=0.1, mod_token_weight=3.0, keep_spliced_per_token=True)
    batch = coll(inst)
    assert len(batch) == 22 and float(batch["concatenated_token_weight"].max()) == 3.0
    model = LlavaLlamaForCausalLM(dims(), "cuda", hf_state=params)
    eng = DPOStepEngine(model.policy, lr=1e-3, total_steps=4, constant_lr=True, dpo_token_weighted=True)
    m = eng.train_step(dict(batch), optimizer_step=False)
    md = eng.metrics_dict(m)
    torch.cuda.synchronize()
    # --- the same arithmetic with the oracle's (bf16-order) per-token log-probs ---
    pb = {k: v.to(torch.bfloat16) for k, v in params.items()}
    ids, labels = batch["concatenated_input_ids"], batch["concatenated_labels"]
    with torch.no_grad():
        ob = O.policy_logps(pb, c, ids, labels, batch["images"].to(torch.bfloat16))
    src, T = ob["src"], ob["labels"].shape[1]
    tw = batch["concatenated_token_weight"].float()
    w_sp = torch.ones(2 * B, T - 1)
    for s_ in range(2 * B):
        for t in range(T - 1):
            j = int(src[s_, t + 1])
            if 1 <= j <= tw.shape[1]:
                w_sp[s_, t] = tw[s_, j - 1]
    mask = (ob["labels"][:, 1:] != -100).float()
    pol_w = (ob["per_token_logps"].float() * w_sp * mask).sum(-1)
    ref_pt = torch.zeros(2 * B, T - 1)
    for kind, off in (("win", 0), ("rej", B)):
        t_ = batch[f"ref_{kind}_per_token_logp_spliced"]
        n = min(T - 1, t_.shape[1])
        ref_pt[off:off + B, :n] = t_[:, :n]
    ref_w = (ref_pt * w_sp * mask).sum(-1)
    losses, cr, rj = O.dpo_loss(pol_w[:B], pol_w[B:], ref_w[:B], ref_w[B:], 0.1)
    assert abs(md["loss"] - float(losses.mean())) <= 2e-3 * max(1.0, abs(float(losses.mean())))
    assert abs(md["logps_train/chosen"] - float(pol_w[:B].mean())) <= 1e-3 * abs(float(pol_w[:B].mean()))
    assert abs(md["logps_train/ref_rejected"] - float(ref_w[B:].mean())) <= 1e-5 * abs(float(ref_w[B:].mean()))
    # --- all weights 1 == the unweighted engine (gradients too) ---
    coll1 = DataCollatorForDPODataset(tokenizer=Tok(), beta=0.1, mod_token_weight=1.0, keep_spliced_per_token=True)
    b1 = coll1(inst)
    mask_rows = (ob["labels"][:, 1:] != -100).float()
    b1["ref_win_logp"] = (ref_pt[:B] * mask_rows[:B]).sum(-1)
    b1["ref_rej_logp"] = (ref_pt[B:] * mask_rows[B:]).sum(-1)
    model.policy.store.grad.zero_()
    mw = eng.train_step(dict(b1), optimizer_step=False).clone()
    gw = model.policy.store.grad.float().clone()
    eng_plain = DPOStepEngine(model.policy, lr=1e-3, total_steps=4, constant_lr=True)
    model.policy.store.grad.zero_()
    mp = eng_plain.train_step(dict(b1), optimizer_step=False).clone()
    gp = model.policy.store.grad.float()
    torch.cuda.synchronize()
    assert abs(float(mw[0]) - float(mp[0])) <= 1e-5 * max(1.0, abs(float(mp[0])))
    assert float((gw - gp).norm() / gp.norm()) <= 1e-3
