"""Optimizer checkpoints across layouts (``internevo_b200/checkpoint/optimizer_interchange.py``): a run resumes exactly with
another ZeRO / data-parallel size, hands its optimizer state to the reference's parameter-wise file layout and takes it back."""
import os
import sys

import pytest
import torch

from common import build_trainer, run_distributed, synthetic_batch, tiny_config

ROWS = 4      # micro-batches per step over the whole job


def _step(trainer, cfg, dp, dpr, seed):
    from internevo_b200.core.context import ParallelMode, global_context as gpc

    T = cfg["data"]["seq_len"] * cfg["data"]["micro_bsz"]
    data, labels = synthetic_batch(ROWS, T, cfg["model"]["vocab_size"], seed=seed)
    per = ROWS // dp
    data = {k: v[dpr * per:(dpr + 1) * per] for k, v in data.items()}
    trainer.zero_grad()
    out = trainer.execute_schedule((data, labels[dpr * per:(dpr + 1) * per]), forward_only=False, return_loss=True,
                                   return_output_label=False)
    ok, _ = trainer.step()
    assert ok
    loss = out[2].detach().clone().reshape(1).float()
    if dp > 1:
        torch.distributed.all_reduce(loss, group=gpc.get_group(ParallelMode.DATA))
        loss /= dp
    return float(loss)


def _run(rank, world, folder, phase, zero1, fmt):
    from internevo_b200.checkpoint import CheckpointManager
    from internevo_b200.core.context import ParallelMode, global_context as gpc
    from internevo_b200.core.trainer import TrainState

    cfg = tiny_config(zero1=zero1, num_layers=2, micro_num=ROWS // world, hidden=64)
    cfg["ckpt"] = dict(enable_save_ckpt=True, save_ckpt_folder=f"local:{folder}", checkpoint_every=2, oss_snapshot_freq=0,
                       auto_resume=(phase == "resume"), async_upload=False, optimizer_ckpt_format=fmt)
    trainer, opt, model, _ = build_trainer(cfg)
    dp, dpr = gpc.get_world_size(ParallelMode.DATA), gpc.get_local_rank(ParallelMode.DATA)
    ts = TrainState(gpc.config, None)
    mm = CheckpointManager(ckpt_config=gpc.config.ckpt, model=model, optimizer=opt, lr_scheduler=trainer.engine._lr_scheduler,
                           model_config=gpc.config.model)
    mm.try_resume_training(ts)
    losses = {}
    if phase == "first":
        for step in (1, 2):
            ts.batch_count = step - 1
            losses[step] = _step(trainer, cfg, dp, dpr, step)
            ts.step_count += 1
            mm.try_save_checkpoint(ts)
        mm.wait_async_upload_finish()
    else:
        assert ts.step_count == 2
    for step in (3, 4):
        losses[step] = _step(trainer, cfg, dp, dpr, step)
    return losses


@pytest.mark.parametrize("save,load", [((2, 2), (1, 1)), ((1, 1), (2, 2)), ((2, 2), (2, 1))],
                         ids=["zero2_to_1rank", "1rank_to_zero2", "zero2_to_replicated"])
def test_resume_with_another_zero_size_is_exact(tmp_path, save, load):
    """(world, zero1 size) at save → at load: the optimizer files are re-sharded through the per-parameter form.  The reference
    refuses this (``hybrid_zero_optim.py:900`` "TODO: Need to take into account the change in the number of DP")."""
    first = run_distributed(_run, save[0], str(tmp_path), "first", save[1], "internevo_b200")
    resumed = run_distributed(_run, load[0], str(tmp_path), "resume", load[1], "internevo_b200")
    for step in (3, 4):    # another reduction order over the data-parallel ranks: equal to rounding
        assert abs(first[0][step] - resumed[0][step]) < 2e-6 * max(1.0, abs(first[0][step])), (first[0], resumed[0])


def _check_reference_files(folder, world):
    """What the reference's ``HybridZeroOptimizer.load_state_dict`` reads (``hybrid_zero_optim.py:899-936``)."""
    model_file = torch.load(os.path.join(folder, "2", "model_tp0_pp0.pt"), weights_only=False)
    numel = {k: v.numel() for k, v in model_file.items()}
    seen = []
    for z in range(world):
        st = torch.load(os.path.join(folder, "2", f"optimizer_tp0_pp0_zo{z}.pt"), weights_only=False)
        assert {"grad_scaler", "base_optim_states", "flat_fp32_weights", "zero_devide_optim_plan"} <= set(st)
        groups = st["base_optim_states"]["param_groups"]
        # an fp32 model: the reference files every fp32 parameter under its "fp32" group (id 1), "default" stays empty
        assert [g["name"] for g in groups] == ["default", "fp32"] and groups[0]["params"] == [] and groups[1]["params"] == [0]
        assert {"lr", "betas", "eps", "weight_decay"} <= set(groups[1])
        assert st["zero_devide_optim_plan"][0] == [[] for _ in range(world)]
        plan = st["zero_devide_optim_plan"][1]
        assert len(plan) == world
        flat, state = st["flat_fp32_weights"][1], st["base_optim_states"]["state"][0]
        want = sum(int(torch.Size([int(d) for d in pid.split("_")[1:]]).numel()) for pid in plan[z])
        assert flat.dtype == torch.float32 and flat.numel() == want == state["exp_avg"].numel() == state["exp_avg_sq"].numel()
        assert float(state["step"]) == 2.0
        seen += [int(pid.split("_")[0]) for pid in plan[z]]
    # every parameter exactly once, numbered by descending size
    assert sorted(seen) == list(range(len(numel)))
    sizes = sorted(numel.values(), reverse=True)
    for z in range(world):
        for pid in torch.load(os.path.join(folder, "2", f"optimizer_tp0_pp0_zo{z}.pt"), weights_only=False)[
                "zero_devide_optim_plan"][1][z]:
            pos, dims = int(pid.split("_")[0]), [int(d) for d in pid.split("_")[1:]]
            assert int(torch.Size(dims).numel()) == sizes[pos]


def test_reference_format_round_trip_is_exact(tmp_path):
    """``ckpt.optimizer_ckpt_format = "reference"`` writes the reference's layout (one flat buffer of whole parameters per ZeRO
    rank, AdamW state dict, plan ids); resuming detects that layout and converts back: the trajectory continues exactly."""
    first = run_distributed(_run, 2, str(tmp_path), "first", 2, "reference")
    _check_reference_files(str(tmp_path), 2)
    resumed = run_distributed(_run, 2, str(tmp_path), "resume", 2, "internevo_b200")
    for step in (3, 4):
        assert abs(first[0][step] - resumed[0][step]) < 1e-6, (first[0], resumed[0])
    # ... and into a job of another size, as a run that moves over from the reference would
    single = run_distributed(_run, 1, str(tmp_path), "resume", 1, "internevo_b200")
    for step in (3, 4):
        assert abs(first[0][step] - single[0][step]) < 2e-6 * max(1.0, abs(first[0][step])), (first[0], single[0])


def test_partition_matches_the_reference_implementation():
    """``reference_partition`` against the plans of the reference's own ``_partition_param_list`` (run unbound on a stub)."""
    import subprocess

    from common import reference_output

    code = f'''
import sys, types, json, torch
sys.path.insert(0, sys.argv.pop(1))
from internlm.solver.optimizer.hybrid_zero_optim import HybridZeroOptimizer
from internlm.core.context import global_context as gpc
gpc.is_rank_for_log = lambda: False
shapes = json.loads(sys.argv[1])
stub = types.SimpleNamespace(_zero_world_size=[int(sys.argv[2])], params_per_rank_id_dict=[], _overlap_sync_param=False)
params = [torch.nn.Parameter(torch.empty(*s)) for s in shapes]
HybridZeroOptimizer._partition_param_list(stub, 0, {{"params": params}})
print("PLAN" + json.dumps(stub.params_per_rank_id_dict[0]))
'''
    import json

    from internevo_b200.checkpoint.optimizer_interchange import reference_partition

    shapes = [[128, 64], [64], [192, 64], [64, 64], [64], [64], [256, 64], [64, 256], [256, 64], [64], [128, 64], [7, 3]]

    def make(ref, dst):
        plans = {}
        for world in (1, 2, 3, 4):
            r = subprocess.run([sys.executable, "-c", code, ref, json.dumps(shapes), str(world)], capture_output=True, text=True,
                               timeout=300, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
            assert r.returncode == 0, r.stderr[-2000:]
            plans[world] = json.loads([line for line in r.stdout.splitlines() if line.startswith("PLAN")][0][4:])
        json.dump(plans, open(dst, "w"))

    plans = json.load(open(reference_output("partition_plans.json", make)))
    for world in (1, 2, 3, 4):
        theirs = plans[str(world)]
        _, ours = reference_partition(shapes, world)
        assert ours == theirs, (world, ours, theirs)


REFERENCE_FORMAT = dict(ckpt_extra=dict(optimizer_ckpt_format="reference"))


@pytest.mark.parametrize("name,world,kw,moe", [
    ("tp2_dp2", 4, dict(tp=2), False),                                   # one set of files per tensor rank
    ("pp2_dp2", 4, dict(pp=2), False),                                   # ... and per pipeline stage (local layer numbering)
    ("llama2", 2, dict(model_type="LLAMA2"), False),                     # wq / wk / wv in the files, one wqkv in memory
    ("internlm_v1", 2, dict(model_type="INTERNLM"), False),              # biases, Wqkv / out_proj / w1 w2 w3 naming
    ("bf16_fp32_norm", 2, dict(dtype="torch.bfloat16", top_level=dict(use_fp32_norm=True)), False),   # the "fp32" group
    # expert group (bf16: in an fp32 model the reference files the experts under "fp32" as well, before it looks for experts)
    ("moe_ep2", 2, dict(model_type="INTERNLM_MoE", num_experts=4, moe_type="MegaBlock-D", dtype="torch.bfloat16"), True),
])
def test_reference_format_round_trip_for_families_and_layouts(tmp_path, name, world, kw, moe):
    """Save in the reference's optimizer layout, resume from it: the trajectory equals the uninterrupted run for every model
    family's key translation (fused wqkv / w13, biases), per-coordinate files and the extra parameter groups."""
    from test_checkpoint_cpu import _run_layout

    first = run_distributed(_run_layout, world, str(tmp_path), "first", dict(kw, **REFERENCE_FORMAT), moe)
    st = torch.load(os.path.join(str(tmp_path), "2", "optimizer_tp0_pp0_zo0.pt"), weights_only=False)
    assert "base_optim_states" in st and "groups" not in st
    resumed = run_distributed(_run_layout, world, str(tmp_path), "resume", kw, moe)
    for r in range(world):
        for s in (3, 4):
            (la, na), (lb, nb) = first[r][s], resumed[r][s]
            assert (la is None) == (lb is None)
            if la is not None:
                assert abs(la - lb) < 1e-6 * max(1.0, abs(la)), (name, first[r], resumed[r])
            for (ka, va), (kb, vb) in zip(na, nb):
                assert ka == kb and abs(va - vb) < 1e-5 * max(1.0, abs(va)), (name, na, nb)


_REFERENCE_LOADER = r'''
import json, sys, types, torch
ref, folder, world, keys = sys.argv[1], sys.argv[2], int(sys.argv[3]), json.loads(sys.argv[4])
sys.path.insert(0, ref)
from internlm.core.context import global_context as gpc
from internlm.core.context.parallel_context import Config
from internlm.solver.optimizer.hybrid_zero_optim import HybridZeroOptimizer
gpc._config = Config(dict(only_load_lr=False))
gpc.is_rank_for_log = lambda: False
model = torch.load(f"{folder}/model_tp0_pp0.pt", weights_only=False)
params = [torch.nn.Parameter(model[k].float()) for k in keys]          # the reference's model.parameters(), in ITS order
part = types.SimpleNamespace(_zero_world_size=[world, world], params_per_rank_id_dict=[[]], _overlap_sync_param=False)
per_rank, _ = HybridZeroOptimizer._partition_param_list(part, 1, {"params": params})      # fp32 model: everything is in group 1
class Scaler:
    def load_state_dict(self, st): self.st = st
for z in range(world):
    weights = torch.cat([p.detach().reshape(-1) for p in per_rank[z]])
    flat = torch.zeros_like(weights).requires_grad_()                   # the rank's fp32 master buffer, to be filled by the load
    low = torch.zeros_like(weights)
    optim = torch.optim.AdamW([dict(params=[], name="default"), dict(params=[flat], name="fp32")], lr=1.0)
    me = types.SimpleNamespace(
        grad_scaler=Scaler(), optim=optim, _fp32_flat_param_groups_of_current_rank={1: flat}, _zero_local_rank=[z, z],
        param_group_no_params_ranks=[set(range(world)), set()], _fp16_param_groups=[[], per_rank[z]],
        _param_store=types.SimpleNamespace(get_flat_fp16_param_by_rank_group=lambda rank, group_id: low),
        params_per_rank_id_dict=None)
    HybridZeroOptimizer.load_state_dict(me, torch.load(f"{folder}/optimizer_tp0_pp0_zo{z}.pt", weights_only=False))
    # an fp32 run: the master weights ARE the weights - the reference now holds, parameter by parameter, what its model file says
    assert torch.equal(flat.detach(), weights) and torch.equal(low, weights), z
    st = optim.state_dict()["state"][0]
    assert st["exp_avg"].shape == weights.shape and float(st["exp_avg"].abs().sum()) > 0 and float(st["step"]) == 2.0
    assert optim.param_groups[1]["lr"] != 1.0 and me.params_per_rank_id_dict is not None and "_scale" in me.grad_scaler.st
print("REFERENCE_LOADED_OK")
'''


def test_the_references_own_loader_accepts_the_exported_files(tmp_path):
    """Files written with ``optimizer_ckpt_format="reference"`` go through the REFERENCE's ``HybridZeroOptimizer.load_state_dict``
    (run unbound on a stub that carries what its ``__init__`` would have built: the parameter partition from its own
    ``_partition_param_list``, one flat fp32 buffer + ``torch.optim.AdamW`` per rank).  torch validates the AdamW state dict, the
    reference its buffer shapes, and afterwards its master buffer equals the weights of its model file parameter by parameter -
    which pins the parameter order and the ``w13`` → ``w1`` / ``w3`` translation.  The files the reference accepted are stored;
    the files exported here must equal them."""
    import json
    import shutil
    import subprocess

    from common import assert_close, reference_output
    from internevo_b200.checkpoint.optimizer_interchange import _reference_order

    run_distributed(_run, 2, str(tmp_path), "first", 2, "reference")
    folder = os.path.join(str(tmp_path), "2")
    files = ("model_tp0_pp0.pt", "optimizer_tp0_pp0_zo0.pt", "optimizer_tp0_pp0_zo1.pt")

    def make(ref, dst):
        keys = _reference_order(list(torch.load(os.path.join(folder, "model_tp0_pp0.pt"), weights_only=False).keys()))
        r = subprocess.run([sys.executable, "-c", _REFERENCE_LOADER, ref, folder, "2", json.dumps(keys)], capture_output=True,
                           text=True, timeout=600, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
        assert r.returncode == 0 and "REFERENCE_LOADED_OK" in r.stdout, r.stderr[-3000:]
        os.makedirs(dst, exist_ok=True)
        for fn in files:
            shutil.copy(os.path.join(folder, fn), dst)

    accepted = reference_output("optimizer_files_accepted", make)
    for fn in files:
        assert_close(torch.load(os.path.join(folder, fn), weights_only=False),
                     torch.load(os.path.join(accepted, fn), weights_only=False), fn)
