"""ORACLE TOOLING — records the reference's own `LLaVA15DPOTrainer.compute_loss` on the rebound seam
(INTEGRATION.md §1) as tests/golden/trainer/compute_loss_seam.npz.

    python oracle/gen_golden_trainer_seam.py [--out DIR]        (needs a CUDA device and oracle/_ref staged)

The reference's compute_loss (muffin/train/trainers.py:279-311), imported from the staged oracle/_ref copy, runs with
only `get_beta_and_logps` and `dpo_loss` rebound to this repo's, on the batch that
tests/test_gpu_trainer_compat.py builds (tiny model, two ragged pairs). Its `loss.backward()` drives the hand-written
backward. The fixture stores the returned loss, the metrics it logs, and the gradient that backward leaves in the
parameter store (its L2 norm and a fixed, seeded sample of 65536 entries), together with the batch's ids and labels.
test_reference_compute_loss_text_on_rebound_seam holds the fused engine to these numbers, so the check runs where the
reference is not installed.
"""
import argparse
import importlib.util
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

SAMPLE = 65536
METRICS = ("rewards_train/chosen", "rewards_train/rejected", "rewards_train/accuracies", "rewards_train/margins",
           "logps_train/chosen", "logps_train/rejected", "logps_train/ref_chosen", "logps_train/ref_rejected")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "tests", "golden", "trainer"))
    args = ap.parse_args()
    from oracle import llava_dpo_oracle as O
    from oracle import stage_ref
    if not stage_ref.available():
        raise SystemExit("oracle/_ref is not staged: run oracle/stage_ref.py where the reference tree exists")
    stage_ref.import_reference()
    import muffin.train.trainers as T
    import rlaifv_b200.trainers as B
    from rlaifv_b200.collator import DataCollatorForDPODataset
    from rlaifv_b200.llava_model import LlavaLlamaForCausalLM
    spec = importlib.util.spec_from_file_location("_trainer_compat", os.path.join(REPO, "tests",
                                                                                  "test_gpu_trainer_compat.py"))
    tc = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tc)

    params = O.make_params(O.TINY, seed=0, scale=0.4)
    model = LlavaLlamaForCausalLM(tc.dims(), "cuda", hf_state=params)
    batch = DataCollatorForDPODataset(tokenizer=tc.Tok(), beta=0.1, mod_token_weight=1.0)(tc.instances(2, seed=3))
    saved = (T.get_beta_and_logps, T.dpo_loss)
    T.get_beta_and_logps, T.dpo_loss = B.get_beta_and_logps, B.dpo_loss            # <- the rebinding
    try:
        logged = []
        stub = SimpleNamespace(args=SimpleNamespace(past_index=-1, dpo_use_average=False, dpo_token_weighted=False,
                                                    task="DPO"),
                               _nested_gather=lambda x: x.reshape(1), log=logged.append)
        model.policy.store.grad.zero_()
        loss = T.LLaVA15DPOTrainer.compute_loss(stub, model, {k: (v.clone() if torch.is_tensor(v) else v)
                                                              for k, v in batch.items()})
        loss.backward()
        model.policy.finalize_embed_grad()
        torch.cuda.synchronize()
    finally:
        T.get_beta_and_logps, T.dpo_loss = saved
    grad = model.policy.store.grad.float()
    g = torch.Generator().manual_seed(0)
    idx = torch.randperm(grad.numel(), generator=g)[:SAMPLE].sort().values
    fx = dict(params_checksum=np.float64(O.params_checksum(params)),
              concatenated_input_ids=batch["concatenated_input_ids"].numpy(),
              concatenated_labels=batch["concatenated_labels"].numpy(),
              loss=np.float64(float(loss.detach())),
              grad_norm=np.float64(float(grad.double().norm())),
              grad_index=idx.numpy().astype(np.int32),
              grad_sample=grad[idx.cuda()].cpu().numpy())
    for k in METRICS:
        fx["metric:" + k] = np.float64(float(logged[0][k]))
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "compute_loss_seam.npz")
    np.savez_compressed(path, **fx)
    print("loss %.8f, grad norm %.6e; written %s" % (fx["loss"], fx["grad_norm"], path))


if __name__ == "__main__":
    main()
