"""Differential tests against the UNMODIFIED reference: ``tests/differential_probe.py`` - written only against the reference's import
paths and signatures - runs with this repository, whose ``internlm`` package is an alias of ``internevo_b200``, and its results are
compared with what the same probe computed with the reference first on ``sys.path``.  The reference's results are stored under
``tests/golden/reference``; ``INTERNEVO_REFERENCE=<checkout of the reference> pytest tests/test_reference_differential_cpu.py``
computes them afresh from the reference and rewrites them.  Everything a loss curve depends on outside the
kernels is compared value by value: sampler batches (ramp-up, epoch roll-over, resume), tokenized-file reading, both packed
datasets item by item, collate functions, learning-rate / beta2 schedules, the dynamic loss scaler, the reported TFLOPS and the
layer partition."""
import json
import math
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from common import assert_close, reference_output

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROBE = os.path.join(ROOT, "tests", "differential_probe.py")


def _probe(script, *args, cwd, timeout=600, **env):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", script), *map(str, args)], capture_output=True, text=True,
                       timeout=timeout, cwd=str(cwd), env=dict(os.environ, CUDA_VISIBLE_DEVICES="", **env))
    assert r.returncode == 0 and "PROBE_OK" in r.stdout, f"{script} {args}: {r.stderr[-3000:]}"


@pytest.fixture(scope="module")
def both(tmp_path_factory):
    import sentencepiece as spm

    work = tmp_path_factory.mktemp("differential")
    rng = np.random.RandomState(1)
    words = ["alpha", "beta", "gamma", "delta", "epsilon", "zeta", "eta", "theta", "iota", "kappa"]
    corpus = work / "corpus.txt"
    corpus.write_text("\n".join(" ".join(rng.choice(words, rng.randint(3, 40))) for _ in range(120)))
    spm.SentencePieceTrainer.Train(input=str(corpus), model_prefix=str(work / "tok"), vocab_size=64, bos_id=1, eos_id=2, unk_id=0,
                                   pad_id=-1, model_type="bpe", minloglevel=2)
    os.makedirs(work / "en")
    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "tokenizer.py"), "--text_input_path", str(corpus),
                    "--bin_output_path", str(work / "en" / "part0.bin"), "--tokenizer_model", str(work / "tok.model")],
                   check=True, capture_output=True)
    ref = reference_output("probe.json", lambda root, dst: _probe(PROBE, root, work, dst, cwd=work))
    _probe(PROBE, ROOT, work, work / "ours.json", cwd=work)
    return json.load(open(ref)), json.load(open(work / "ours.json"))


def _same(a, b, tol=0.0):
    if isinstance(a, dict):
        return isinstance(b, dict) and a.keys() == b.keys() and all(_same(a[k], b[k], tol) for k in a)
    if isinstance(a, (list, tuple)):
        return isinstance(b, (list, tuple)) and len(a) == len(b) and all(_same(x, y, tol) for x, y in zip(a, b))
    if isinstance(a, float) or isinstance(b, float):
        return abs(a - b) <= tol * max(1.0, abs(a))
    return a == b


@pytest.mark.parametrize("key", ["sampler_plain", "sampler_rank1", "sampler_rampup", "sampler_resume", "sampler_state_keys"])
def test_static_batch_sampler_yields_the_references_batches(both, key):
    ref, ours = both
    assert _same(ref[key], ours[key]), (key, ref[key][:3], ours[key][:3])


@pytest.mark.parametrize("key", ["jsonl_len", "jsonl_items", "pack_into_one", "pack_with_cut", "packed_collate", "jsonl_collate",
                                 "unpack"])
def test_data_pipeline_items_equal_the_references(both, key):
    """Item by item, every pack of both packed datasets: tokens, labels (incl. what happens to the label of a token whose sample
    continues in the next pack: predicted across the cut by ``PackedDatasetWithCut``, ignored by the pack-into-one form),
    ``cu_seqlens``, position ``indexes`` and type ids."""
    ref, ours = both
    assert _same(ref[key], ours[key]), key


@pytest.mark.parametrize("key", ["beta2", "scaler", "flops", "partition"])
def test_schedules_scaler_flops_and_partition_equal_the_references(both, key):
    ref, ours = both
    assert _same(ref[key], ours[key], tol=1e-12), (key, ref[key], ours[key])


@pytest.mark.parametrize("key,total,init,ratio,eta", [("lr_cos", 400, 0, 0.05, 1e-5), ("lr_cos_init", 400, 7, 0.1, 1e-4)])
def test_learning_rate_schedule(both, key, total, init, ratio, eta):
    """Ours is the closed form: 0 for ``init_steps``, linear warm-up, then ``eta + (lr - eta) (1 + cos(pi t / T)) / 2``.  The
    reference chains torch's RECURSIVE ``CosineAnnealingLR.get_lr``; with the torch of this image the recursion starts from
    ``last_epoch = 0`` without torch's former special case, which multiplies its whole cosine by ``2 / (1 + cos(pi / T))``
    (1 + 1.7e-5 here, 1 + 2e-9 for a 50k-step run) - the two agree to that factor and exactly on warm-up."""
    ref, ours = both
    base, warm = 1e-3, int(total * ratio) + init
    T = total - warm
    for i in range(total):
        want = 0.0 if i < init else (i + 1 - init) / (warm - init) * base if i < warm else \
            eta + (base - eta) * (1 + math.cos(math.pi * (i - warm) / T)) / 2
        assert abs(ours[key][i] - want) < 1e-15, (i, ours[key][i], want)
    assert _same(ref[key][:warm], ours[key][:warm], tol=1e-12)
    excess = 2 / (1 + math.cos(math.pi / T)) - 1
    assert max(abs(a - b) for a, b in zip(ref[key][:total], ours[key][:total])) <= excess * base * 1.01


@pytest.mark.parametrize("config", ["7B_sft", "7B_internlm2", "7B_isp_sft", "7B_MoE4_sft", "7B_llama2"])
def test_args_sanity_check_fills_a_reference_config_like_the_reference(tmp_path, config):
    """A config file SHIPPED BY THE REFERENCE goes through ``args_sanity_check`` on both sides: every default it fills in, every
    derived key (``sequence_parallel``, ``packed_length``, checkpoint sub-keys, monitor section, MoE / ISP switches ...) comes
    out identical - the configuration a reference user brings along means the same thing here."""
    def make_input(root, dst):
        code = ("import json, sys; sys.path.insert(0, sys.argv[1]); from internlm.core.context.parallel_context import Config; "
                "json.dump(dict(Config.from_file(sys.argv[2])), open(sys.argv[3], 'w'), indent=1, sort_keys=True)")
        subprocess.run([sys.executable, "-c", code, root, os.path.join(root, "configs", config + ".py"), dst], check=True,
                       cwd=str(tmp_path), env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))

    src = reference_output(f"config_{config}.json", make_input)
    out = {}
    for side, root in (("reference", None), ("ours", ROOT)):
        dst = str(tmp_path / f"{side}.json")
        if root is None:
            dst = reference_output(f"config_{config}.checked.json",
                                   lambda root, dst: _probe("differential_config_probe.py", root, src, dst, cwd=tmp_path))
        else:
            _probe("differential_config_probe.py", root, src, dst, cwd=tmp_path)
        out[side] = json.load(open(dst))

    def flat(d, prefix=""):
        res = {}
        for k, v in d.items():
            res.update(flat(v, prefix + k + ".") if isinstance(v, dict) else {prefix + k: v})
        return res

    a, b = flat(out["reference"]), flat(out["ours"])
    diff = {k: (a.get(k, "<absent>"), b.get(k, "<absent>")) for k in sorted(set(a) | set(b)) if a.get(k, "<absent>") != b.get(k, "<absent>")}
    assert not diff, diff


def test_skip_batches_and_top2_gating_equal_the_references(both):
    """``top2gating`` (capacity, second-expert masking, renormalised weights, drops, l_aux) agrees entry by entry of the
    ``[token, expert, slot]`` combine tensor, with and without token dropping."""
    ref, ours = both
    assert ref["skipper"] == ours["skipper"]
    for key in ("gate_top2", "gate_top2_drop"):
        assert _same(ref[key], ours[key], tol=1e-6), key


@pytest.mark.parametrize("key", ["gate_top1", "gate_top1_drop"])
def test_top1_gating_without_random_token_selection(both, key):
    """Same auxiliary loss, expert counts and capacity, every kept token weighted with its gate probability at a slot of its own.
    WHICH tokens of an over-subscribed expert are kept is not compared: without random token selection the reference takes
    ``torch.topk`` of a 0 / 1 mask, i.e. whatever order topk gives equal elements; this framework keeps the earliest tokens."""
    import torch

    ref, ours = both
    assert abs(ref[key]["l_aux"] - ours[key]["l_aux"]) < 1e-6 and ref[key]["counts"] == ours[key]["counts"]
    probs = torch.tensor(ours["gate_probs"])
    kept = []
    for side in (ref, ours):
        combine = torch.tensor(side[key]["combine"])
        assert combine.shape == torch.tensor(ref[key]["combine"]).shape            # same capacity
        tok, exp, slot = combine.nonzero(as_tuple=True)
        assert torch.allclose(combine[tok, exp, slot], probs[tok, exp], atol=1e-6)
        assert (exp == probs.argmax(1)[tok]).all() and len(set(zip(exp.tolist(), slot.tolist()))) == len(tok)
        kept.append(torch.bincount(exp, minlength=4).tolist())
    assert kept[0] == kept[1] == [min(c, torch.tensor(ref[key]["combine"]).shape[2]) for c in ref[key]["counts"]]


def _model_probe(family, cwd):
    return reference_output(f"model_{family}.pt", lambda root, dst: _probe("differential_model_probe.py", root, family, dst, cwd=cwd))


def _our_logits(rank, world, family, ref_file):
    import torch

    from common import build_trainer, tiny_config

    ref = torch.load(ref_file, weights_only=False)
    kw = dict(model_type=family, num_layers=2, hidden=32, heads=4, kv_heads=2, vocab=64, seq_len=16, micro_bsz=2, micro_num=1)
    cfg = tiny_config(**kw)
    cfg["model"].update(parallel_output=False, use_flash_attn=False)
    cfg["data"]["use_packed_dataset"] = False
    if family == "INTERNLM_MoE":
        cfg["model"].update(num_experts=4, moe_use_residual=False, moe_type="GShard")
        cfg["moe"] = dict(top_k=1, capacity_factor=4.0, eval_capacity_factor=4.0, min_capacity=4, noisy_gate_policy=None,
                          drop_tokens=True, use_rts=False)
        cfg["loss"]["moe_loss_coeff"] = 0.1
    _, _, model, _ = build_trainer(cfg)
    inner = model.model
    missing, unexpected = inner.load_state_dict(ref["state"], strict=False)
    assert not missing and not unexpected, (missing, unexpected)      # the reference's state dict IS a state dict of ours
    inner.eval()
    with torch.no_grad():
        out = model(input_ids=ref["ids"])
    moe = None
    if family == "INTERNLM_MoE":
        out, moe = out
        moe = [float(x) for x in moe]
    return out.float().reshape(-1, out.shape[-1]), ref["logits"].reshape(-1, ref["logits"].shape[-1]), moe, ref["moe_losses"]


@pytest.mark.parametrize("family", ["INTERNLM", "INTERNLM2_PUBLIC", "LLAMA2", "INTERNLM_MoE"])
def test_model_forward_equals_the_references_on_its_own_weights(tmp_path, family):
    """The reference builds the model (its torch attention / rotary / norm path on CPU) and runs a forward; its ``state_dict()`` is
    loaded into this framework's model of the same family - no key is missing or unexpected - and the logits agree to fp32
    rounding: parameter layout (interleaved GQA ``wqkv``, ``w1`` / ``w3`` fused into ``w13``, biases), RoPE convention, norms, MLP
    and the GShard MoE block (gate, capacity, combine, auxiliary loss) compute the same function.  The MoE case routes top-1 with
    room for every token: the reference's top-2 gate picks the second expert with Gumbel noise and its top-1 gate drops by
    ``topk`` tie order, neither of which two separately seeded processes can reproduce (the gates themselves are compared on
    equal RNG state above)."""
    from common import run_distributed

    dst = _model_probe(family, tmp_path)
    ours, theirs, moe, their_moe = run_distributed(_our_logits, 1, family, dst)[0]
    assert ours.shape == theirs.shape
    assert float((ours - theirs).abs().max()) < 2e-6 * max(1.0, float(theirs.abs().max())), float((ours - theirs).abs().max())
    if family == "INTERNLM_MoE":
        assert len(moe) == len(their_moe) and all(abs(a - b) < 1e-6 for a, b in zip(moe, their_moe)), (moe, their_moe)


def _our_training(rank, world, ref_file, family="INTERNLM2_PUBLIC"):
    import torch

    import internevo_b200 as fw
    from common import tiny_config
    from internevo_b200.initialize import initialize_distributed_env
    from internevo_b200.models.losses import FlashGPTLMLoss
    from internevo_b200.train import get_scheduler_hooks, initialize_model, initialize_optimizer

    ref = torch.load(ref_file, weights_only=False)
    ref["final"] = torch.load(ref_file[:-3] + ".final.pt", weights_only=False)
    S, MB, MN = 16, 2, 2
    cfg = tiny_config(model_type=family, num_layers=2, hidden=32, heads=4, kv_heads=2, vocab=64, seq_len=S, micro_bsz=MB,
                      micro_num=MN)
    cfg["model"].update(parallel_output=False, use_flash_attn=False)
    if family == "INTERNLM_MoE":
        cfg["model"].update(num_experts=4, moe_use_residual=False, moe_type="GShard")
        cfg["moe"] = dict(top_k=1, capacity_factor=4.0, eval_capacity_factor=4.0, min_capacity=4, noisy_gate_policy=None,
                          drop_tokens=True, use_rts=False)
        cfg["loss"]["moe_loss_coeff"] = 0.1
    cfg["data"].update(use_packed_dataset=False, total_steps=10)
    cfg["adam"].update(lr=3e-3, adam_eps=1e-4, weight_decay=0.01)
    cfg["lr_scheduler"].update(total_steps=2000, warmup_ratio=0.001, eta_min=1e-4)
    cfg["grad_scaler"]["fp16"]["initial_scale"] = 2**16
    cfg["hybrid_zero_optimizer"]["clip_grad_norm"] = 100.0
    initialize_distributed_env(config=cfg, launcher="torch", seed=1024)
    model = initialize_model()
    model.model.load_state_dict(ref["state"], strict=True)
    opt, b2, lrs = initialize_optimizer(model)
    crit = FlashGPTLMLoss(parallel_output=False, label_smoothing=0)
    trainer, _, _, _ = fw.initialize_trainer(model=model, optimizer=opt, criterion=crit, lr_scheduler=lrs, beta2_scheduler=b2,
                                             scheduler_hooks=get_scheduler_hooks(None, opt, None))
    trainer.train()
    losses, norms = [], []
    for ids, labels in ref["batches"]:
        cu = torch.arange(0, MB * S + 1, S, dtype=torch.int32).repeat(MN, 1)
        idx = torch.arange(S).repeat(MN, MB)
        trainer.zero_grad()
        out = trainer.execute_schedule(({"input_ids": ids.clone(), "cu_seqlens": cu, "indexes": idx}, labels.clone()),
                                       forward_only=False, return_loss=True, return_output_label=False)
        ok, gn = trainer.step()
        assert ok
        losses.append(float(out[2]))
        norms.append(sum(float(v) ** 2 for v in gn.values()) ** 0.5)
    final = model.model.state_dict()
    drift = max(float((final[k] - ref["final"][k]).abs().max()) for k in ref["final"])
    moved = max(float((ref["final"][k] - ref["state"][k]).abs().max()) for k in ref["final"])
    ref_norms = [sum(float(v) ** 2 for v in n.values()) ** 0.5 for n in ref["norms"]]
    return losses, ref["losses"], norms, ref_norms, drift, moved


@pytest.mark.parametrize("family", ["INTERNLM2_PUBLIC", "INTERNLM", "LLAMA2", "INTERNLM_MoE"])
def test_eight_training_steps_follow_the_reference(tmp_path, family):
    """The reference's own training loop (``initialize_model`` → ``HybridZeroOptimizer`` over ``torch.optim.AdamW`` →
    ``initialize_trainer`` → non-pipeline scheduler with two accumulated micro-batches of un-packed sequences → torch cross entropy)
    runs 8 optimizer steps on CPU; this framework starts from the same weights, sees the same batches and must produce the same
    loss and gradient norm at every step and the same weights at the end - loss scaling, accumulation, AdamW with decoupled decay
    and bias correction, warm-up and cosine learning rate, the fp32 master copy.
    Two properties of the reference are side-stepped, not imitated: (1) gradient clipping is configured out of reach - for an
    fp32 model the reference files every parameter under its ``fp32`` group and then indexes the per-group clip factors by the
    position among NON-EMPTY groups (``hybrid_zero_optim.py:863-876``), i.e. it takes the factor of the empty ``default`` group
    and never clips, while bf16 runs (groups aligned) clip like this framework; (2) the schedule is long, so the factor
    ``2 / (1 + cos(pi / T))`` that torch's recursive cosine puts on the reference's learning rate is below 1e-5."""
    import torch

    from common import run_distributed

    def make(root, dst):
        # the final weights in a file of their own: no stored file is larger than 1 MB
        _probe("differential_train_probe.py", root, dst, family, cwd=tmp_path, timeout=900)
        ref = torch.load(dst, weights_only=False)
        torch.save(ref.pop("final"), dst[:-3] + ".final.pt")
        torch.save(ref, dst)

    dst = reference_output(f"train_{family}.pt", make)
    losses, ref_losses, norms, ref_norms, drift, moved = run_distributed(_our_training, 1, dst, family)[0]
    assert len(losses) == len(ref_losses) == 8
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) < 2e-6 * max(1.0, abs(b)), (losses, ref_losses)
    for a, b in zip(norms, ref_norms):
        assert abs(a - b) < 3e-5 * max(1.0, abs(b)), (norms, ref_norms)
    # the weights moved by ~lr per step; ours ended where the reference's did.  (Adam divides by |g|: fp32 rounding of small
    # gradient entries - different summation orders, a fused w13 GEMM - shows up as a per-entry update difference of up to ~1 % of
    # the learning rate; ``adam_eps = 1e-4`` keeps entries whose gradient is pure rounding noise, like the key bias of the
    # InternLM-v1 attention whose true gradient is zero, from random-walking by +-lr per step on either side.)
    assert moved > 5e-3 and drift < 0.03 * moved, (drift, moved)


def _resume_reference_checkpoint(rank, world, ref_file, folder):
    import torch

    import internevo_b200 as fw
    from common import tiny_config
    from internevo_b200.checkpoint import CheckpointManager
    from internevo_b200.core.context import global_context as gpc
    from internevo_b200.core.trainer import TrainState
    from internevo_b200.initialize import initialize_distributed_env
    from internevo_b200.models.losses import FlashGPTLMLoss
    from internevo_b200.train import get_scheduler_hooks, initialize_model, initialize_optimizer

    ref = torch.load(ref_file, weights_only=False)
    S, MB, MN = 16, 2, 2
    cfg = tiny_config(num_layers=2, hidden=32, heads=4, kv_heads=2, vocab=64, seq_len=S, micro_bsz=MB, micro_num=MN)
    cfg["model"].update(parallel_output=False, use_flash_attn=False)
    cfg["data"].update(use_packed_dataset=False, total_steps=10)
    cfg["adam"].update(lr=3e-3, adam_eps=1e-4, weight_decay=0.01)
    cfg["lr_scheduler"].update(total_steps=2000, warmup_ratio=0.001, eta_min=1e-4)
    cfg["grad_scaler"]["fp16"]["initial_scale"] = 2**16
    cfg["hybrid_zero_optimizer"]["clip_grad_norm"] = 100.0
    cfg["ckpt"] = dict(enable_save_ckpt=False, auto_resume=False,
                       load_ckpt_info=dict(path=f"local:{folder}/4", content=("model", "optimizer", "scheduler"),
                                           ckpt_type="internevo"))
    initialize_distributed_env(config=cfg, launcher="torch", seed=77)       # another seed: every weight must come from the files
    model = initialize_model()
    opt, b2, lrs = initialize_optimizer(model)
    crit = FlashGPTLMLoss(parallel_output=False, label_smoothing=0)
    trainer, _, _, _ = fw.initialize_trainer(model=model, optimizer=opt, criterion=crit, lr_scheduler=lrs, beta2_scheduler=b2,
                                             scheduler_hooks=get_scheduler_hooks(None, opt, None))
    trainer.train()
    ts = TrainState(gpc.config, None)
    CheckpointManager(ckpt_config=gpc.config.ckpt, model=model, optimizer=opt, lr_scheduler=lrs,
                      model_config=gpc.config.model).try_resume_training(ts)
    assert ts.step_count == 4, ts.step_count
    # the position in the schedule: the reference's warm-up wrapper stopped counting at 2, its cosine scheduler counted 2 more
    their_sched = torch.load(f"{folder}/4/schedulder.pt", weights_only=False)
    assert (their_sched["last_epoch"], their_sched["after_scheduler_dict"]["last_epoch"]) == (2, 2) and lrs.last_epoch == 4
    # (equal up to the factor 2 / (1 + cos(pi / T)) = 1 + 6e-7 of the reference's recursive cosine, see test_learning_rate_schedule)
    assert abs(opt.param_groups[0]["lr"] - their_sched["_last_lr"][0]) < 2e-6 * their_sched["_last_lr"][0]
    losses = []
    for ids, labels in ref["batches"][4:]:
        cu = torch.arange(0, MB * S + 1, S, dtype=torch.int32).repeat(MN, 1)
        idx = torch.arange(S).repeat(MN, MB)
        trainer.zero_grad()
        out = trainer.execute_schedule(({"input_ids": ids.clone(), "cu_seqlens": cu, "indexes": idx}, labels.clone()),
                                       forward_only=False, return_loss=True, return_output_label=False)
        ok, _ = trainer.step()
        assert ok
        losses.append(float(out[2]))
    final = model.model.state_dict()
    drift = max(float((final[k] - ref["final"][k]).abs().max()) for k in ref["final"])
    moved = max(float((ref["final"][k] - ref["state"][k]).abs().max()) for k in ref["final"])
    return losses, ref["losses"][4:], drift, moved


def test_a_checkpoint_written_by_the_reference_resumes_here(tmp_path):
    """The reference trains 4 steps on CPU and ITS ``CheckpointManager`` writes a checkpoint (``model_tp0_pp0.pt``,
    ``optimizer_tp0_pp0_zo0.pt`` in its parameter-wise flat layout, ``schedulder.pt``, ``context.pt``), then trains 4 more steps.
    This framework - initialised with another seed - loads model, optimizer and scheduler state from those files and its next 4
    steps reproduce the reference's: weights, fp32 master copy, Adam moments and step count, loss scale and the position in the
    learning-rate schedule all arrive through the files (``checkpoint/optimizer_interchange.py``)."""
    from common import run_distributed

    def make(root, dst):
        shutil.rmtree(dst, ignore_errors=True)
        os.makedirs(dst)
        _probe("differential_train_probe.py", root, os.path.join(dst, "train.pt"), "INTERNLM2_PUBLIC", os.path.join(dst, "ckpt"),
               cwd=tmp_path, timeout=900)
        for fn in os.listdir(os.path.join(dst, "ckpt")):      # only the checkpoint after step 4 is resumed
            if fn not in ("4", "4.step"):
                shutil.rmtree(os.path.join(dst, "ckpt", fn), ignore_errors=True)

    base = reference_output("checkpoint_from_reference", make)
    dst, folder = os.path.join(base, "train.pt"), os.path.join(base, "ckpt")
    assert {"model_tp0_pp0.pt", "optimizer_tp0_pp0_zo0.pt", "schedulder.pt", "context.pt", "4.step"} <= set(os.listdir(f"{folder}/4"))
    losses, ref_losses, drift, moved = run_distributed(_resume_reference_checkpoint, 1, dst, folder)[0]
    assert len(losses) == 4
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) < 2e-6 * max(1.0, abs(b)), (losses, ref_losses)
    assert moved > 5e-3 and drift < 0.03 * moved, (drift, moved)


def _train_and_save_for_the_reference(rank, world, folder):
    import torch

    import internevo_b200 as fw
    from common import tiny_config
    from internevo_b200.checkpoint import CheckpointManager
    from internevo_b200.core.context import global_context as gpc
    from internevo_b200.core.trainer import TrainState
    from internevo_b200.initialize import initialize_distributed_env
    from internevo_b200.models.losses import FlashGPTLMLoss
    from internevo_b200.train import get_scheduler_hooks, initialize_model, initialize_optimizer

    S, MB, MN = 16, 2, 2
    cfg = tiny_config(num_layers=2, hidden=32, heads=4, kv_heads=2, vocab=64, seq_len=S, micro_bsz=MB, micro_num=MN)
    cfg["model"].update(parallel_output=False, use_flash_attn=False)
    cfg["data"].update(use_packed_dataset=False, total_steps=10)
    cfg["adam"].update(lr=3e-3, adam_eps=1e-4, weight_decay=0.01)
    cfg["lr_scheduler"].update(total_steps=2000, warmup_ratio=0.001, eta_min=1e-4)
    cfg["grad_scaler"]["fp16"]["initial_scale"] = 2**16
    cfg["hybrid_zero_optimizer"]["clip_grad_norm"] = 100.0
    cfg["ckpt"] = dict(enable_save_ckpt=True, save_ckpt_folder=f"local:{folder}", checkpoint_every=4, oss_snapshot_freq=0,
                       auto_resume=False, async_upload=False, optimizer_ckpt_format="reference")
    initialize_distributed_env(config=cfg, launcher="torch", seed=5)
    model = initialize_model()
    opt, b2, lrs = initialize_optimizer(model)
    crit = FlashGPTLMLoss(parallel_output=False, label_smoothing=0)
    trainer, _, _, _ = fw.initialize_trainer(model=model, optimizer=opt, criterion=crit, lr_scheduler=lrs, beta2_scheduler=b2,
                                             scheduler_hooks=get_scheduler_hooks(None, opt, None))
    trainer.train()
    ts = TrainState(gpc.config, None)
    mm = CheckpointManager(ckpt_config=gpc.config.ckpt, model=model, optimizer=opt, lr_scheduler=lrs, model_config=gpc.config.model)
    g = torch.Generator().manual_seed(7)        # the batch stream of differential_train_probe.py
    losses = []
    for step in range(8):
        ids = torch.randint(1, 64, (MN, MB * S), generator=g)
        labels = torch.cat([ids[:, 1:], torch.full((MN, 1), -100)], 1)
        labels[:, S - 1::S] = -100
        cu = torch.arange(0, MB * S + 1, S, dtype=torch.int32).repeat(MN, 1)
        idx = torch.arange(S).repeat(MN, MB)
        trainer.zero_grad()
        out = trainer.execute_schedule(({"input_ids": ids, "cu_seqlens": cu, "indexes": idx}, labels), forward_only=False,
                                       return_loss=True, return_output_label=False)
        ok, _ = trainer.step()
        assert ok
        losses.append(float(out[2]))
        if step < 4:
            ts.batch_count, ts.step_count = step, ts.step_count + 1
            mm.try_save_checkpoint(ts)
    mm.wait_async_upload_finish()
    return losses, {k: v.clone() for k, v in model.model.state_dict().items()}


def test_the_reference_resumes_a_checkpoint_written_here(tmp_path):
    """The other direction with the reference's real code: this framework trains 4 steps and saves with
    ``optimizer_ckpt_format="reference"``; the reference's ``CheckpointManager.try_resume_training`` loads model, optimizer
    (``HybridZeroOptimizer.load_state_dict`` + ``torch.optim.AdamW.load_state_dict``) and scheduler from that folder on CPU and its
    next 4 steps reproduce the 4 steps this framework went on to take."""
    import torch

    from common import run_distributed

    folder = str(tmp_path / "our_ckpt")
    losses, final = run_distributed(_train_and_save_for_the_reference, 1, folder)[0]

    def make(root, dst):
        shutil.rmtree(dst, ignore_errors=True)
        shutil.copytree(os.path.join(folder, "4"), os.path.join(dst, "loaded", "4"))
        _probe("differential_train_probe.py", root, os.path.join(dst, "resumed.pt"), "INTERNLM2_PUBLIC", os.path.join(dst, "loaded"),
               "resume", cwd=tmp_path, timeout=900)

    base = reference_output("checkpoint_for_reference", make)
    # the files written here are the ones the reference was shown to load
    for fn in ("model_tp0_pp0.pt", "optimizer_tp0_pp0_zo0.pt", "schedulder.pt"):
        assert_close(torch.load(os.path.join(folder, "4", fn), weights_only=False),
                      torch.load(os.path.join(base, "loaded", "4", fn), weights_only=False), fn)
    theirs = torch.load(os.path.join(base, "resumed.pt"), weights_only=False)
    assert len(theirs["losses"]) == 4
    for a, b in zip(theirs["losses"], losses[4:]):
        assert abs(a - b) < 2e-6 * max(1.0, abs(b)), (theirs["losses"], losses[4:])
    drift = max(float((final[k] - theirs["final"][k]).abs().max()) for k in final)
    assert drift < 2e-4, drift


@pytest.fixture(scope="module")
def data_folder(tmp_path_factory):
    import sentencepiece as spm

    work = tmp_path_factory.mktemp("loader")
    rng = np.random.RandomState(3)
    words = ["alpha", "beta", "gamma", "delta", "epsilon", "zeta", "eta", "theta", "iota", "kappa"]
    (work / "corpus.txt").write_text("\n".join(" ".join(rng.choice(words, 12)) for _ in range(300)))
    spm.SentencePieceTrainer.Train(input=str(work / "corpus.txt"), model_prefix=str(work / "tok"), vocab_size=64, bos_id=1,
                                   eos_id=2, unk_id=0, pad_id=-1, model_type="bpe", minloglevel=2)
    for split, lo, hi, n in (("train", 1, 30, 60), ("valid", 25, 60, 40)):      # validation lines long enough for min_length 50
        for lang, files in (("en", 2), ("cn", 1), ("code", 1)):
            os.makedirs(work / "data" / split / lang)
            for i in range(files):
                (work / "c.txt").write_text("\n".join(" ".join(rng.choice(words, rng.randint(lo, hi))) for _ in range(n)))
                subprocess.run([sys.executable, os.path.join(ROOT, "tools", "tokenizer.py"), "--text_input_path", str(work / "c.txt"),
                                "--bin_output_path", str(work / "data" / split / lang / f"part{i}.bin"), "--tokenizer_model",
                                str(work / "tok.model")], check=True, capture_output=True)
    return work


@pytest.mark.parametrize("dp_rank,pack", [(0, "cut"), (1, "cut"), (0, "one")])
def test_train_and_validation_loaders_yield_the_references_batches(data_folder, dp_rank, pack):
    """The data stream of a run: which files form which dataset in which order (the reference concatenates them in the order
    rank 0's ``os.walk`` finds the folders), the type id of every token (position of its sub-folder in the sorted listing), short-
    sample filtering (``min_length`` for training, 50 tokens for validation), packing, the sampler's order and the collated batch -
    the first six training batches and the first two batches of every validation set are identical, tensor by tensor, on both
    data-parallel ranks and in both packing modes."""
    def run(root, dst):
        _probe("differential_loader_probe.py", root, data_folder / "data", dst, *(["one"] if pack == "one" else []), cwd=data_folder,
               PROBE_DP_RANK=str(dp_rank))

    dst = str(data_folder / f"ours_{dp_rank}_{pack}.json")
    run(ROOT, dst)
    out = {"ours": json.load(open(dst)), "reference": json.load(open(reference_output(f"loader_{dp_rank}_{pack}.json", run)))}
    a, b = out["reference"], out["ours"]
    assert a["types"] == b["types"] == ["cn", "code", "en"] and a["len"] == b["len"] > 6
    for i, (x, y) in enumerate(zip(a["batches"], b["batches"])):
        assert x == y, f"training batch {i} differs"
    assert sorted(a["valid"]) == sorted(b["valid"]) == ["cn", "code", "en"] and a["valid"] == b["valid"]


def test_metrics_report_the_references_keys_and_values(tmp_path):
    """Accuracy, perplexity, ``loss_from_metric`` and the per-type ``acc/`` ``tokens/`` ``loss/`` entries of the step log: every key
    the reference's ``AccPerplex`` / ``LossWithTypeId`` return is returned here with the same value (this framework adds
    ``perplexity/<type>``)."""
    def run(root, dst):
        _probe("differential_metric_probe.py", root, dst, cwd=tmp_path)

    run(ROOT, tmp_path / "ours.json")
    out = {"ours": json.load(open(tmp_path / "ours.json")), "reference": json.load(open(reference_output("metrics.json", run)))}
    for part in ("acc", "loss"):
        theirs, ours = out["reference"][part], out["ours"][part]
        assert set(theirs) <= set(ours), (part, sorted(set(theirs) - set(ours)))
        for k, v in theirs.items():
            assert abs(v - ours[k]) < 1e-4 * max(1.0, abs(v)), (k, v, ours[k])


def _small_tokenizer_model(cwd):
    """A small SentencePiece model (the reference's own is 1.6 MB) on which both code bases' tokenizer tools run."""
    def make(root, dst):
        import sentencepiece as spm

        rng = np.random.RandomState(11)
        words = ["alpha", "beta", "gamma", "delta", "epsilon", "zeta", "eta", "theta", "iota", "kappa", "训练", "模型", "数据"]
        (cwd / "spm.txt").write_text("\n".join(" ".join(rng.choice(words, rng.randint(1, 30))) for _ in range(400)))
        spm.SentencePieceTrainer.Train(input=str(cwd / "spm.txt"), model_prefix=str(cwd / "spm"), vocab_size=96, bos_id=1,
                                       eos_id=2, unk_id=0, pad_id=-1, model_type="bpe", character_coverage=1.0,
                                       normalization_rule_name="identity", minloglevel=2)
        shutil.copy(cwd / "spm.model", dst)

    return reference_output("tokenizer_small.model", make)


def test_tokenizer_tool_writes_the_references_bytes(tmp_path):
    """``tools/tokenizer.py`` of both code bases on the same text with the same SentencePiece model: the ``.bin`` files are
    byte-identical and the ``.meta`` offsets / lengths equal (kept int64 here - the reference's int32 wraps beyond 2 GiB)."""
    model = _small_tokenizer_model(tmp_path)
    rng = np.random.RandomState(5)
    words = ["alpha", "beta", "gamma", "delta", "epsilon", "zeta", "eta", "theta", "iota", "kappa", "训练", "模型", "数据"]
    text = tmp_path / "corpus.txt"
    text.write_text("\n".join(" ".join(rng.choice(words, rng.randint(1, 40))) for _ in range(200)))
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")

    def make(root, dst):
        # the reference's tool reads the model next to itself and its tokenizer class from ../transformers
        os.makedirs(tmp_path / "ref" / "tools")
        shutil.copy(os.path.join(root, "tools", "tokenizer.py"), tmp_path / "ref" / "tools")
        shutil.copy(model, tmp_path / "ref" / "tools" / "tokenizer_internlm.model")
        os.symlink(os.path.join(root, "transformers"), tmp_path / "ref" / "transformers")
        r = subprocess.run([sys.executable, str(tmp_path / "ref" / "tools" / "tokenizer.py"), "--text_input_path", str(text),
                            "--bin_output_path", dst + ".bin"], capture_output=True, text=True, timeout=600, cwd=str(tmp_path), env=env)
        assert r.returncode == 0, r.stderr[-2000:]
        os.replace(dst + ".bin", dst)

    ref = reference_output("tokenizer.bin", make)
    ref_meta = reference_output("tokenizer.bin.meta", lambda root, dst: os.replace(ref + ".bin.meta", dst))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "tokenizer.py"), "--text_input_path", str(text),
                        "--bin_output_path", str(tmp_path / "ours.bin"), "--tokenizer_model", model], capture_output=True, text=True,
                       timeout=600, cwd=str(tmp_path), env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    assert open(ref, "rb").read() == open(tmp_path / "ours.bin", "rb").read()
    a, b = np.load(ref_meta, allow_pickle=True), np.load(tmp_path / "ours.bin.meta", allow_pickle=True)
    assert a.shape == b.shape and (a == b).all()


def _our_evaluation(rank, world, ref_file, data):
    import torch

    import internevo_b200 as fw
    from common import tiny_config
    from internevo_b200.data import build_valid_loader_with_data_type
    from internevo_b200.eval.evaluation import evaluate_on_val_dls
    from internevo_b200.initialize import initialize_distributed_env
    from internevo_b200.models.losses import FlashGPTLMLoss
    from internevo_b200.train import get_scheduler_hooks, initialize_model, initialize_optimizer

    ref = torch.load(ref_file, weights_only=False)
    cfg = tiny_config(num_layers=2, hidden=32, heads=4, kv_heads=2, vocab=64, seq_len=16, micro_bsz=2, micro_num=2)
    cfg["model"].update(parallel_output=False, use_flash_attn=False)
    cfg["data"].update(use_packed_dataset=False, total_steps=10, valid_every=1, valid_micro_num=2, valid_folder=os.path.join(data, "valid"))
    initialize_distributed_env(config=cfg, launcher="torch", seed=3)
    model = initialize_model()
    model.model.load_state_dict(ref["state"], strict=True)
    opt, b2, lrs = initialize_optimizer(model)
    crit = FlashGPTLMLoss(parallel_output=False, label_smoothing=0)
    trainer, _, _, _ = fw.initialize_trainer(model=model, optimizer=opt, criterion=crit, lr_scheduler=lrs, beta2_scheduler=b2,
                                             scheduler_hooks=get_scheduler_hooks(None, opt, None))
    scalars = {}

    class Writer:
        def add_scalar(self, key, value, step):
            scalars[key] = float(value)

    class Logger:
        def info(self, *a, **k):
            pass

        warning = error = info

    val_dls = build_valid_loader_with_data_type()
    evaluate_on_val_dls(trainer, val_dls, Writer(), Logger(), step_count=3)
    return scalars, {k: len(v) for k, v in val_dls.items()}, ref["scalars"], ref["sizes"]


def test_validation_reports_the_references_numbers(data_folder, tmp_path):
    """``evaluate_on_val_dls`` of both code bases on the same weights and the same validation folder (three sub-folders): the same
    validation sets with the same number of batches, and per set the same ``val/<name>_loss`` / ``_acc`` / ``_plex`` scalars."""
    from common import run_distributed

    dst = reference_output("eval.pt", lambda root, dst: _probe("differential_eval_probe.py", root, dst, data_folder / "data",
                                                               cwd=tmp_path, timeout=900))
    ours, sizes, theirs, their_sizes = run_distributed(_our_evaluation, 1, dst, str(data_folder / "data"))[0]
    assert sizes == their_sizes and sorted(sizes) == ["cn", "code", "en"]
    keys = {k for k in theirs if k != "step"}
    assert keys == {k for k in ours if k != "step"} and len(keys) == 9
    for k in keys:
        # accuracy / perplexity are reported rounded to 4 decimals: a value on a rounding boundary may land one step apart
        tol = 1.01e-4 if k.endswith(("_acc", "_plex")) else 1e-6 * max(1.0, abs(theirs[k]))
        assert abs(ours[k] - theirs[k]) <= tol, (k, ours[k], theirs[k])


@pytest.mark.parametrize("family", ["internlm2", "internlm"])
def test_hf_remote_code_equals_the_references(tmp_path, family):
    """The Hugging Face model code shipped next to converted weights (``huggingface/<family>_model``) against the reference's
    (``transformers/<family>_model``, the code on the hub): a model created by the reference's class saves its ``state_dict``, ours
    loads it without a missing or unexpected key and computes the same logits."""
    import torch

    def make(root, dst):
        os.makedirs(dst, exist_ok=True)
        _probe("differential_hf_probe.py", "ref", os.path.join(root, "transformers", f"{family}_model"), family,
               os.path.join(dst, "m"), cwd=tmp_path)

    theirs = reference_output(f"hf_{family}", make)
    prefix = str(tmp_path / family)
    shutil.copy(os.path.join(theirs, "m.weights"), prefix + ".weights")
    # ours the way ``tools/convert2hf.py::install_remote_code`` puts it next to converted weights: one flat folder (the v1 files
    # import the shared helpers from the InternLM2 files)
    flat = tmp_path / "remote_code"
    os.makedirs(flat)
    for sub in ("internlm2_model", f"{family}_model"):
        for fn in os.listdir(os.path.join(ROOT, "huggingface", sub)):
            if fn.endswith(".py") and fn != "__init__.py":
                src = open(os.path.join(ROOT, "huggingface", sub, fn)).read().replace("from ..internlm2_model.", "from .")
                (flat / fn).write_text(src)
    _probe("differential_hf_probe.py", "ours", flat, family, prefix, cwd=tmp_path)
    a, b = torch.load(os.path.join(theirs, "m.ref.logits")), torch.load(prefix + ".ours.logits")
    assert a.shape == b.shape and float((a - b).abs().max()) < 2e-6 * max(1.0, float(a.abs().max()))


def test_converted_checkpoint_scores_like_the_training_model_in_the_references_hf_class(tmp_path):
    """End to end across both code bases: the reference's TRAINING model (CPU, torch attention) produces weights and logits;
    ``tools/convert2hf.py`` of this repository converts the checkpoint folder; the reference's HF class
    (``transformers/internlm2_model``) loads the result and returns the training model's logits - the converter (GQA ``wqkv``
    un-interleaving, rotary row permutation, names) is right with respect to both ends of the reference."""
    import torch
    from safetensors.torch import load_file

    dst = _model_probe("INTERNLM2_PUBLIC", tmp_path)
    probe = torch.load(dst, weights_only=False)
    ckpt = tmp_path / "ckpt"
    os.makedirs(ckpt)
    torch.save(probe["state"], ckpt / "model_tp0_pp0.pt")
    torch.save(dict(hidden_size=32, num_layers=2, num_attention_heads=4, num_kv_attention_heads=2, vocab_size=64, mlp_ratio=2,
                    layer_norm_epsilon=1e-5, no_bias=True, embed_split_hidden=True, norm_type="rmsnorm", dtype=torch.float32),
               ckpt / "model_config.pt")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "convert2hf.py"), "--src", str(ckpt), "--tgt", str(tmp_path / "hf"),
                        "--dtype", "float32"], capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    weights = {}
    for fn in os.listdir(tmp_path / "hf"):
        if fn.endswith(".safetensors"):
            weights.update(load_file(str(tmp_path / "hf" / fn)))
    def make(root, dst):
        os.makedirs(dst, exist_ok=True)
        torch.save(weights, os.path.join(dst, "conv.hf_weights"))
        torch.save(probe["ids"], os.path.join(dst, "conv.ids"))
        _probe("differential_hf_probe.py", "load", os.path.join(root, "transformers", "internlm2_model"), "internlm2",
               os.path.join(dst, "conv"), cwd=tmp_path)

    base = reference_output("converted_internlm2", make)
    # the converter's output is what the reference's HF class was shown to load
    assert_close(weights, torch.load(os.path.join(base, "conv.hf_weights")), "hf_weights")
    hf_logits, train_logits = torch.load(os.path.join(base, "conv.load.logits")), probe["logits"]
    assert hf_logits.shape == train_logits.shape
    assert float((hf_logits - train_logits).abs().max()) < 2e-6 * max(1.0, float(train_logits.abs().max()))


def test_reverted_hf_model_scores_alike_in_the_references_training_model(tmp_path):
    """The way back: a model of the reference's HF class -> ``tools/revert_hf.py`` -> the reference's TRAINING model loads the
    resulting ``model_tp0_pp0.pt`` key for key and returns the HF model's logits."""
    import torch
    from safetensors.torch import save_file

    env = dict(PROBE_INTERMEDIATE="256", PROBE_MLP_RATIO="8")

    def make(root, dst):
        os.makedirs(dst, exist_ok=True)
        _probe("differential_hf_probe.py", "ref", os.path.join(root, "transformers", "internlm2_model"), "internlm2",
               os.path.join(dst, "hf"), cwd=tmp_path, **env)

    theirs = reference_output("hf_internlm2_mlp8", make)
    hf_dir = tmp_path / "hf_model"
    os.makedirs(hf_dir)
    weights = {k: v.contiguous() for k, v in torch.load(os.path.join(theirs, "hf.weights")).items() if "inv_freq" not in k}
    save_file(weights, str(hf_dir / "model.safetensors"))
    json.dump(dict(hidden_size=32, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2, vocab_size=64,
                   intermediate_size=256, rms_norm_eps=1e-5, rope_theta=10000, bias=False, model_type="internlm2",
                   architectures=["InternLM2ForCausalLM"]), open(hf_dir / "config.json", "w"))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "revert_hf.py"), "--src", str(hf_dir), "--tgt", str(tmp_path / "ckpt"),
                        "--tp_size", "1", "--embed_split"], capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    torch.manual_seed(1)
    ids = torch.randint(1, 64, (2, 12))          # the ids differential_hf_probe.py scored
    state = torch.load(tmp_path / "ckpt" / "model_tp0_pp0.pt", weights_only=False)

    def make_given(root, dst):
        torch.save({"state": state, "ids": ids}, dst)

    def make_logits(root, dst):
        _probe("differential_model_probe.py", root, "INTERNLM2_PUBLIC", dst, given, cwd=tmp_path, **env)

    given = reference_output("reverted_internlm2.pt", make_given)
    # the reverted checkpoint is the one the reference's training model was shown to load
    assert_close(state, torch.load(given, weights_only=False)["state"], "model_tp0_pp0.pt")
    train_logits = torch.load(reference_output("reverted_internlm2.logits.pt", make_logits), weights_only=False)["logits"]
    hf_logits = torch.load(os.path.join(theirs, "hf.ref.logits"))
    assert train_logits.shape == hf_logits.shape
    assert float((train_logits - hf_logits).abs().max()) < 2e-6 * max(1.0, float(hf_logits.abs().max()))


def test_alpaca_tokenizer_writes_the_references_bytes(tmp_path):
    """``tools/alpaca_tokenizer.py`` of both code bases on the same instruction data: chat template, negated prompt tokens, end-of-
    turn ids, truncation and the train / validation split give byte-identical ``dataset.bin`` files."""
    model = _small_tokenizer_model(tmp_path)
    rng = np.random.RandomState(0)
    words = ["alpha", "beta", "gamma", "delta", "epsilon", "zeta", "数据", "模型"]
    data = [{"instruction": " ".join(rng.choice(words, 5)), "input": " ".join(rng.choice(words, 3)) if i % 2 else "",
             "output": " ".join(rng.choice(words, rng.randint(3, 2500 if i == 7 else 12)))} for i in range(60)]   # one over-long answer
    json.dump(data, open(tmp_path / "alpaca.json", "w"))
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")

    def run(tool, out):
        r = subprocess.run([sys.executable, tool, str(tmp_path / "alpaca.json"), out, model, "--split_ratio", "0.1"],
                           capture_output=True, text=True, timeout=600, cwd=str(tmp_path), env=env)
        assert r.returncode == 0, r.stderr[-2000:]

    run(os.path.join(ROOT, "tools", "alpaca_tokenizer.py"), str(tmp_path / "ours"))
    ref = reference_output("alpaca", lambda root, dst: run(os.path.join(root, "tools", "alpaca_tokenizer.py"), dst))
    for split in ("train", "valid"):
        a = open(os.path.join(ref, split, "en", "dataset.bin"), "rb").read()
        b = open(tmp_path / "ours" / split / "en" / "dataset.bin", "rb").read()
        assert a == b and len(a) > 0, split
