"""The reference's module tree resolves through the ``internlm`` alias, and the small public helpers that came with it
behave (reference paths cited next to each implementation)."""
import ast
import importlib
import json
import math
import os
import sys

import pytest
import torch

from common import ROOT, reference_output, run_distributed  # noqa: F401

# by design: one accelerator backend
NO_COUNTERPART = {"internlm.accelerator.npu_accelerator"}


def _reference_modules(root, dst):
    """Every module of the reference's ``internlm`` package with the public classes / functions it defines."""
    tree, out = os.path.join(root, "internlm"), {}
    for d, _, fs in sorted(os.walk(tree)):
        for f in sorted(fs):
            if f.endswith(".py"):
                path = os.path.join(d, f)
                mod = os.path.relpath(path, root)[:-3].replace(os.sep, ".")
                mod = mod[:-9] if mod.endswith(".__init__") else mod
                out[mod] = [node.name for node in ast.parse(open(path).read()).body
                            if isinstance(node, (ast.ClassDef, ast.FunctionDef)) and not node.name.startswith("_")]
    json.dump(out, open(dst, "w"), indent=0)


def test_every_reference_module_path_resolves():
    modules = json.load(open(reference_output("modules.json", _reference_modules)))
    missing, names, absent = [], 0, 0
    for mod, public in modules.items():
        if mod in NO_COUNTERPART:
            continue
        try:
            m = importlib.import_module(mod)
        except Exception as e:  # noqa: BLE001
            missing.append((mod, repr(e)[:80]))
            continue
        names += len(public)
        absent += sum(not hasattr(m, name) for name in public)
    assert not missing, missing
    # every public class / function of the reference is reachable under its own name
    assert names > 300 and absent == 0, (names, absent)


def test_lr_schedulers():
    from internlm.solver.schedulers.lr_scheduler import CosineAnnealingWarmupLR, WarmupScheduler

    p = [torch.nn.Parameter(torch.zeros(1))]
    opt = torch.optim.SGD(p, lr=1.0)
    s = CosineAnnealingWarmupLR(opt, total_steps=20, warmup_steps=4, eta_min=0.1)
    lrs = []
    for _ in range(20):
        lrs.append(opt.param_groups[0]["lr"])
        s.step()
    assert lrs[:4] == [0.25, 0.5, 0.75, 1.0] and lrs[4] == 1.0
    assert abs(lrs[12] - (0.1 + 0.9 * (1 + math.cos(math.pi * 8 / 16)) / 2)) < 1e-9 and min(lrs[4:]) > 0.1

    opt = torch.optim.SGD(p, lr=1.0)
    w = WarmupScheduler(opt, 4, torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=10))
    lrs = []
    for _ in range(9):
        lrs.append(opt.param_groups[0]["lr"])
        w.step()
    assert lrs[:4] == [0.25, 0.5, 0.75, 1.0] and abs(lrs[6] - (1 + math.cos(math.pi * 2 / 10)) / 2) < 1e-6
    state = w.state_dict()
    assert state["after_scheduler_type"] == "CosineAnnealingLR"
    w.load_state_dict(state)


def test_optimizer_tensor_list_helpers():
    from internlm.solver.optimizer.base_optimizer import BaseOptimizer
    from internlm.solver.optimizer.utils import (
        BaseGradScaler,
        calc_lp,
        flatten,
        get_norm,
        has_inf_or_nan,
        release_param_grad,
        split_half_float_double,
        sync_param,
        unflatten,
    )

    torch.manual_seed(0)
    g = [torch.randn(5), torch.randn(3, 2), torch.randn(4).double()]
    flat = flatten(g[:2])
    assert flat.numel() == 11 and all(torch.equal(a, b) for a, b in zip(unflatten(flat, g[:2]), g[:2]))
    assert [len(b) for b in split_half_float_double(g)] == [2, 1]
    assert abs(float(get_norm(g[:2], 2.0)) - float(flat.norm() ** 2)) < 1e-4
    assert abs(float(calc_lp(g[:2], 3.0)) - float(flat.abs().pow(3).sum())) < 1e-4
    assert float(get_norm(g[:2], math.inf)) == float(flat.abs().max())
    assert has_inf_or_nan(torch.tensor([1.0, float("inf")])) and has_inf_or_nan(torch.tensor([float("nan")]))
    assert not has_inf_or_nan(flat)
    params = [torch.nn.Parameter(t.clone()) for t in g[:2]]
    sync_param(flat, params)
    flat.zero_()
    assert all(float(p.detach().abs().sum()) == 0 for p in params)            # they alias the flat buffer now
    for p in params:
        p.grad = torch.ones_like(p)
    release_param_grad(params)
    assert all(p.grad is None for p in params)
    s = BaseGradScaler(128.0)
    s.update(True)
    assert s.scale == 128.0 and s.inv_scale == 1 / 128 and s.state_dict() == {"scale": 128.0}

    lin = torch.nn.Linear(4, 4)
    opt = BaseOptimizer(torch.optim.SGD(lin.parameters(), lr=0.5))
    before = lin.weight.detach().clone()
    opt.zero_grad()
    opt.backward(lin(torch.ones(2, 4)).sum())
    opt.step()
    assert not torch.equal(before, lin.weight) and opt.param_groups[0]["lr"] == 0.5 and "state" in opt.state_dict()


def test_metric_scatter_norm_and_attention_oracles():
    from internlm.model.metrics import vanilla_scatter
    from internlm.model.modules.multi_head_attention import CrossAttention, DistributedAttention, SelfAttention
    from internlm.model.modules.mlp import FeedForward, get_mlp_cls
    from internlm.model.ops.norm import RMSNormTorch, manual_rms_norm
    from internlm.model.utils import Silu

    src, idx = torch.tensor([1.0, 2.0, 3.0, 4.0]), torch.tensor([0, 2, 0, 2])
    assert vanilla_scatter(src, idx, dim=0, dim_size=4).tolist() == [4.0, 0.0, 6.0, 0.0]
    assert vanilla_scatter(torch.ones(2, 3), torch.tensor([1, 1, 0]), dim=1).tolist() == [[1.0, 2.0], [1.0, 2.0]]

    torch.manual_seed(0)
    x, n = torch.randn(3, 5, 16), RMSNormTorch(16, eps=1e-6)
    with torch.no_grad():
        n.weight.uniform_(0.5, 1.5)
    want = x / x.pow(2).mean(-1, keepdim=True).add(1e-6).sqrt() * n.weight
    assert torch.allclose(n(x), want, atol=1e-6) and torch.allclose(manual_rms_norm(x, (16,), None, 1e-6) * n.weight, want, atol=1e-6)
    a, b = torch.randn(4, 8), torch.randn(4, 8)
    assert torch.allclose(Silu(a, b), torch.nn.functional.silu(a) * b)
    assert all(get_mlp_cls(m) is FeedForward for m in ("mtp", "msp", "fsp", "isp"))

    sdpa = torch.nn.functional.scaled_dot_product_attention
    qkv = torch.randn(2, 7, 3, 4, 8)
    want = sdpa(*[t.transpose(1, 2) for t in qkv.unbind(2)], is_causal=True).transpose(1, 2)
    assert torch.allclose(SelfAttention(causal=True)(qkv), want, atol=1e-5)
    assert torch.allclose(DistributedAttention(SelfAttention(causal=True), None)(qkv=qkv), want, atol=1e-5)
    keep = torch.ones(2, 7, dtype=torch.bool)
    keep[:, 5:] = False
    got = SelfAttention()(qkv, key_padding_mask=keep)
    want = sdpa(*[t.transpose(1, 2) for t in qkv.unbind(2)], attn_mask=keep[:, None, None, :]).transpose(1, 2)
    assert torch.allclose(got, want, atol=1e-5)
    q, kv = torch.randn(2, 1, 4, 8), torch.randn(2, 7, 2, 2, 8)       # one decode step against a 7-token GQA cache
    k, v = [t.repeat_interleave(2, 2).transpose(1, 2) for t in kv.unbind(2)]
    assert torch.allclose(CrossAttention(causal=True)(q, kv), sdpa(q.transpose(1, 2), k, v).transpose(1, 2), atol=1e-5)


def test_legacy_checkpoint_config_keys():
    from internlm.initialize.legacy.launch import auto_resume_sanity_check, ckpt_info_sanity_check

    assert auto_resume_sanity_check({}) is True and auto_resume_sanity_check({"load_given_ckpt": True}) is False
    assert ckpt_info_sanity_check({}) is None
    assert ckpt_info_sanity_check({"load_model_only_folder": "local:/m"}) == dict(path="local:/m", content=("model",),
                                                                                  ckpt_type="internlm")
    assert ckpt_info_sanity_check({"load_ckpt_folder": "/c"})["content"] == ("model", "sampler", "optimizer")
    assert ckpt_info_sanity_check({"load_ckpt_folder": "/c", "load_optimizer": False})["content"] == ("model", "sampler")
    with pytest.raises(AssertionError):
        ckpt_info_sanity_check({"load_ckpt_folder": "/c", "load_model_only_folder": "/m"})


def _write_bin(path, n, seed):
    import json

    import numpy as np

    rng, offs, off = np.random.RandomState(seed), [], 0
    with open(path, "wb") as f:
        for _ in range(n):
            line = (json.dumps({"tokens": rng.randint(1, 100, rng.randint(4, 20)).tolist()}) + "\n").encode()
            f.write(line)
            offs.append((off, len(json.loads(line)["tokens"])))
            off += len(line)
    np.save(open(path + ".meta", "wb"), np.array(offs, dtype=np.int64))


def test_validation_sets_per_subfolder(tmp_path):
    from internlm.data.tokenized.dataset import get_dataset_dict
    from internlm.data.utils import get_dataset_type_ids_map

    for name, n in (("zhihu", 9), ("baike", 5)):
        os.makedirs(tmp_path / name)
        _write_bin(str(tmp_path / name / "valid.bin"), n, seed=n)
    _write_bin(str(tmp_path / "zhihu" / "valid2.bin"), 3, seed=1)
    _write_bin(str(tmp_path / "zhihu" / "train.bin"), 7, seed=2)
    d = get_dataset_dict(str(tmp_path), split="valid", min_length=0)
    assert list(d) == ["baike", "zhihu"] and len(d["zhihu"]) == 12 and len(d["baike"]) == 5
    assert len(get_dataset_dict(str(tmp_path), split="", min_length=0)["zhihu"]) == 19
    assert not get_dataset_dict(str(tmp_path), split="valid") or \
        len(get_dataset_dict(str(tmp_path), split="valid")["zhihu"]) < 12      # default: samples under 50 tokens are left out
    assert get_dataset_type_ids_map(str(tmp_path)) == {"baike": 0, "zhihu": 1}


def _valid_loader_worker(rank, world, folder):
    from common import tiny_config

    from internevo_b200.core.context import ParallelMode
    from internevo_b200.core.context import global_context as gpc
    from internevo_b200.data.build_dataloader import build_valid_loader_with_data_type
    from internevo_b200.initialize import initialize_distributed_env

    cfg = tiny_config(micro_bsz=2, micro_num=2)
    cfg["data"].update(valid_folder=folder, valid_micro_num=2, valid_min_length=0)
    initialize_distributed_env(config=cfg, launcher="torch", seed=5)
    dls = build_valid_loader_with_data_type()
    # zhihu: 12 samples / dp 2 = 6 per rank -> batch min(4, 6) = 4; baike: 5 // 2 = 2 -> batch 2; tiny: 1 // 2 = 0 -> skipped
    out = {k: [len(b[1]) for b in dl] for k, dl in dls.items()}
    first = {k: next(iter(dl))[0]["input_ids"][0, :4].tolist() for k, dl in dls.items()}
    return out, first, gpc.get_local_rank(ParallelMode.DATA)


def test_valid_loader_batches_and_rank_split(tmp_path):
    for name, n in (("zhihu", 12), ("baike", 5), ("tiny", 1)):
        os.makedirs(tmp_path / name)
        _write_bin(str(tmp_path / name / "valid.bin"), n, seed=n)
    res = run_distributed(_valid_loader_worker, 2, str(tmp_path))
    for out, _, _ in res:
        assert out == {"baike": [2], "zhihu": [4]}, out
    assert res[0][1]["zhihu"] != res[1][1]["zhihu"], "the two data-parallel ranks must read different samples"


def _ulysses_worker(rank, world):
    import torch.distributed as dist

    from common import tiny_config
    from internevo_b200.core.communication.utils import gather_split_1d_tensor, split_tensor_into_1d_equal_chunks
    from internevo_b200.core.context import ParallelMode
    from internevo_b200.core.context import global_context as gpc
    from internevo_b200.initialize import initialize_distributed_env
    from internevo_b200.models.modules import DistributedAttention, SelfAttention

    initialize_distributed_env(config=tiny_config(tp=2, mode="isp", wp=2), launcher="torch", seed=5)
    group = gpc.get_group(ParallelMode.TENSOR)
    torch.manual_seed(0)
    qkv = torch.randn(2, 8, 3, 4, 8, requires_grad=True)           # full sequence, same on both ranks
    want = SelfAttention(causal=True)(qkv)
    want.square().sum().backward()
    gfull = qkv.grad.clone()
    local = qkv.detach()[:, rank * 4:(rank + 1) * 4].clone().requires_grad_()
    got = DistributedAttention(SelfAttention(causal=True), group)(qkv=local)
    got.square().sum().backward()
    assert torch.allclose(got, want[:, rank * 4:(rank + 1) * 4], atol=1e-5)
    assert torch.allclose(local.grad, gfull[:, rank * 4:(rank + 1) * 4], atol=1e-5)

    t = torch.arange(24.0).view(2, 12)
    part = split_tensor_into_1d_equal_chunks(t)
    assert part.tolist() == list(range(rank * 12, rank * 12 + 12))
    assert torch.equal(gather_split_1d_tensor(part).view(2, 12), t)
    dist.barrier()
    return True


def test_distributed_attention_and_1d_split_two_ranks():
    assert all(run_distributed(_ulysses_worker, 2))


def _custom_ckpt_type_worker(rank, world, folder):
    from common import build_trainer, tiny_config

    from internevo_b200.checkpoint import CheckpointManager
    from internevo_b200.checkpoint.checkpoint_manager import CheckpointLoadMethod
    from internevo_b200.core.context import global_context as gpc
    from internevo_b200.core.trainer import TrainState

    seen = []

    def load_mine(ckpt_mm, load_info, train_state):
        seen.append((load_info["path"], sorted(c for c in ("model", "optimizer") if load_info["content"].need_load(c))))
        return "model, "

    CheckpointLoadMethod.register_ckpt_load_type("mine", load_mine)
    cfg = tiny_config(num_layers=2)
    # old-style keys are translated; an explicit load_ckpt_info wins over them
    cfg["ckpt"] = dict(enable_save_ckpt=False, auto_resume=False, load_ckpt_folder=folder, load_optimizer=False)
    trainer, opt, model, _ = build_trainer(cfg)
    mm = CheckpointManager(ckpt_config=gpc.config.ckpt, model=model, optimizer=opt, lr_scheduler=None, model_config=gpc.config.model)
    legacy = dict(mm.load_ckpt_info)
    assert legacy["path"] == folder and legacy["content"].need_load("model") and legacy["content"].need_load("sampler")
    assert not legacy["content"].need_load("optimizer")
    gpc.config.ckpt["load_ckpt_info"] = dict(path=folder, content=("model",), ckpt_type="mine")
    mm = CheckpointManager(ckpt_config=gpc.config.ckpt, model=model, optimizer=opt, lr_scheduler=None, model_config=gpc.config.model)
    mm.try_resume_training(TrainState(gpc.config, None))
    return seen


def test_custom_checkpoint_type_and_legacy_keys(tmp_path):
    (seen,) = run_distributed(_custom_ckpt_type_worker, 1, str(tmp_path))
    assert seen == [(str(tmp_path), ["model"])]


def _async_p2p_worker(rank, world):
    from common import tiny_config

    from internevo_b200.core.communication.p2p import (
        send_backward_and_recv_next_backward_async,
        send_forward_and_recv_next_forward_async,
    )
    from internevo_b200.initialize import initialize_distributed_env

    initialize_distributed_env(config=tiny_config(pp=2, num_layers=4, micro_num=2), launcher="torch", seed=5)
    shape = torch.Size([3, 4])
    # forward direction: stage 0 sends, stage 1 receives; the work between the two next() calls overlaps the transfer
    co = send_forward_and_recv_next_forward_async(torch.full(shape, 7.0) if rank == 0 else None,
                                                  recv_prev_shape=shape if rank == 1 else None, dtype=torch.float32)
    next(co)
    busy = torch.ones(8).sum()
    got = next(co)
    assert (got is None) if rank == 0 else (torch.equal(got, torch.full(shape, 7.0)) and got.requires_grad)
    # backward direction: stage 1 sends the input gradient, stage 0 receives it
    co = send_backward_and_recv_next_backward_async(torch.full(shape, -2.0) if rank == 1 else None,
                                                    recv_next_shape=shape if rank == 0 else None, dtype=torch.float32)
    next(co)
    got = next(co)
    assert (got is None) if rank == 1 else torch.equal(got, torch.full(shape, -2.0))
    return float(busy)


def test_two_phase_async_p2p_coroutines():
    assert run_distributed(_async_p2p_worker, 2) == [8.0, 8.0]


class _FakeObjectStore:
    """In-memory stand-ins for the ``tos`` and ``oss2`` SDK surfaces the storage clients use."""

    def __init__(self):
        self.blobs = {}                                             # (bucket, key) -> bytes
        store = self

        class _Obj:
            def __init__(self, key):
                self.key = key

        class _Stream:
            def __init__(self, data):
                self._d = data

            def read(self):
                return self._d

        class TosClientV2:
            def __init__(self, ak, sk, endpoint, region, enable_crc=False):
                store.tos_args = (ak, sk, endpoint, region)
                self._mp = {}

            def put_object(self, bucket, key, content=None):
                store.blobs[(bucket, key)] = content.read()

            def get_object(self, bucket, key):
                return _Stream(store.blobs[(bucket, key)])

            def delete_object(self, bucket, key):
                store.blobs.pop((bucket, key), None)

            def list_objects_type2(self, bucket, prefix="", continuation_token=None):
                keys = sorted(k for b, k in store.blobs if b == bucket and k.startswith(prefix))
                start = int(continuation_token or 0)                # two keys per page: exercises the continuation loop
                page = type("R", (), {})()
                page.contents = [_Obj(k) for k in keys[start:start + 2]]
                page.is_truncated = start + 2 < len(keys)
                page.next_continuation_token = str(start + 2)
                return page

            def create_multipart_upload(self, bucket, key):
                self._mp[(bucket, key)] = {}
                return type("R", (), {"upload_id": "u1"})()

            def upload_part(self, bucket, key, upload_id, n, content=None):
                self._mp[(bucket, key)][n] = content.read()
                return n

            def complete_multipart_upload(self, bucket, key, upload_id, parts):
                store.blobs[(bucket, key)] = b"".join(self._mp[(bucket, key)][n] for n in parts)

        class Bucket:
            def __init__(self, auth, endpoint, name, enable_crc=False):
                self.name = name

            def put_object(self, key, data):
                store.blobs[(self.name, key)] = data if isinstance(data, bytes) else data.read()

            def put_object_from_file(self, key, path):
                store.blobs[(self.name, key)] = open(path, "rb").read()

            def get_object(self, key):
                return _Stream(store.blobs[(self.name, key)])

            def delete_object(self, key):
                store.blobs.pop((self.name, key), None)

        def iterator(bucket, prefix=""):
            return iter([_Obj(k) for b, k in sorted(store.blobs) if b == bucket.name and k.startswith(prefix)])

        import types

        self.tos = types.SimpleNamespace(TosClientV2=TosClientV2)
        self.oss2 = types.SimpleNamespace(Auth=lambda ak, sk: (ak, sk), Bucket=Bucket, ObjectIteratorV2=iterator)


@pytest.mark.parametrize("url", ["volc:vc://ckpts.tos-cn-beijing.volces.com/run1", "oss2:ali://ckpts.oss-cn-hangzhou.aliyuncs.com/run1"])
def test_volc_and_ali_object_stores(monkeypatch, tmp_path, url):
    import internevo_b200.utils.storage_manager as sm

    fake = _FakeObjectStore()
    monkeypatch.setitem(sys.modules, "tos", fake.tos)
    monkeypatch.setitem(sys.modules, "oss2", fake.oss2)
    for k in ("VOLC_ACCESS_KEY_ID", "ALI_ACCESS_KEY_ID"):
        monkeypatch.setenv(k, "ak")
    for k in ("VOLC_SECRET_ACCESS_KEY_ID", "ALI_SECRET_ACCESS_KEY_ID"):
        monkeypatch.setenv(k, "sk")
    monkeypatch.setattr(sm.VolcClient, "PART", 1 << 10)             # force the multipart path for the async upload
    sm.check_tmp_folder_accessibility(str(tmp_path / "stage"))
    mgr = sm.StorageManager(True, tmp_local_folder=str(tmp_path / "stage"), async_mode=True)
    state = {"w": torch.arange(2000.0), "step": 7}
    mgr.save(f"{url}/7/model_tp0_pp0.pt", state)                    # asynchronous: staged file + md5 sidecar
    mgr.save(f"{url}/7/context.pt", {"step": 7}, async_upload=False)
    mgr.save(f"{url}/8/context.pt", {"step": 8}, async_upload=False)
    mgr.set_pending_marker(f"{url}/7.step")
    assert not mgr.is_exists(f"{url}/7.step")                       # the marker appears only after the uploads finished
    assert mgr.wait() and mgr.is_exists(f"{url}/7.step")
    assert os.listdir(tmp_path / "stage") == []
    assert mgr.get_fns(url) == ["7", "7.step", "8"]
    assert mgr.get_fns(f"{url}/7") == ["context.pt", "model_tp0_pp0.pt", "model_tp0_pp0.pt.md5"]
    back = mgr.load(f"{url}/7/model_tp0_pp0.pt")
    assert torch.equal(back["w"], state["w"]) and back["step"] == 7
    mgr.delete_obj(f"{url}/8/context.pt")
    assert not mgr.is_exists(f"{url}/8") and mgr.is_exists(f"{url}/7")
    if url.startswith("volc"):
        assert fake.tos_args == ("ak", "sk", "tos-cn-beijing.volces.com", "cn-beijing")
    assert sm.get_mount_point_free_size(str(tmp_path)) > 0


def test_dense_gating_functions_agree_with_the_layer_and_the_einsum_form():
    from internlm.model.moe.gshard_layer import TopKGate, top1gating, top2gating

    torch.manual_seed(0)
    S, h, E = 48, 16, 4
    x = torch.randn(S, h)
    for k in (1, 2):
        gate = TopKGate(h, E, k=k, capacity_factor=1.0, min_capacity=4, use_rts=False)
        logits = torch.nn.functional.linear(x, gate.wg.weight)
        torch.manual_seed(7)
        l_aux, w, ex, sl, keep, cap, counts = gate(x)
        torch.manual_seed(7)                                         # same Gumbel draw for the second expert
        l2, combine, mask, c2 = (top1gating(logits, 1.0, 4, use_rts=False) if k == 1 else top2gating(logits, 1.0, 4))
        assert combine.shape == (S, E, cap) and torch.equal(c2, counts) and torch.allclose(l2, l_aux)
        assert mask.sum(0).max() <= 1, "one token per (expert, slot)"
        assert mask.sum((1, 2)).max() <= k and int(mask.sum()) == int(keep.sum())
        assert mask.sum((0, 2)).max() <= cap
        # dense dispatch / combine einsums (GShard) == index scatter / gather used by the layer
        dispatched = torch.einsum("sec,sm->ecm", mask.float(), x)
        rows = (ex * cap + sl)[keep]
        tok = torch.arange(S).unsqueeze(1).expand(S, k)[keep]
        want = torch.zeros(E * cap, h).index_copy(0, rows, x[tok]).view(E, cap, h)
        assert torch.allclose(dispatched, want)
        y = torch.randn(E, cap, h)
        combined = torch.einsum("sec,ecm->sm", combine, y)
        want = torch.zeros(S, h).index_add_(0, tok, y.view(E * cap, h)[rows] * w[keep].unsqueeze(1))
        assert torch.allclose(combined, want, atol=1e-6)
        if k == 2:
            kept_both = keep.all(1)
            assert torch.allclose(combine.sum((1, 2))[kept_both], torch.ones(int(kept_both.sum())), atol=1e-6)
