"""Spawn-N-processes harness (CPU/gloo or GPU/NCCL), mirroring the reference's test strategy
(``tests/test_core/utils.py:149-159``, ``tests/common_fixture.py:108-123``) with a CPU variant."""
import os
import socket
import sys
import traceback

import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


GOLDEN = os.path.join(ROOT, "tests", "golden", "reference")
REFERENCE = os.environ.get("INTERNEVO_REFERENCE")


def reference_output(name, make):
    """Path of what the reference computed for ``name``, stored under ``tests/golden/reference``.  With ``INTERNEVO_REFERENCE``
    set to a checkout of the reference, ``make(reference_root, path)`` runs the reference and stores its result there first."""
    path = os.path.join(GOLDEN, name)
    if REFERENCE:
        os.makedirs(os.path.dirname(path), exist_ok=True)
        make(REFERENCE, path)
    assert os.path.exists(path), path
    return path


def assert_close(a, b, where):
    """``a`` equals ``b`` key by key, tensors to float rounding (computed on another CPU, in another order)."""
    if isinstance(a, dict):
        assert isinstance(b, dict) and sorted(a, key=str) == sorted(b, key=str), (where, sorted(a, key=str), sorted(b, key=str))
        for k in a:
            assert_close(a[k], b[k], f"{where}/{k}")
    elif isinstance(a, (list, tuple)):
        assert isinstance(b, (list, tuple)) and len(a) == len(b), where
        for i, (x, y) in enumerate(zip(a, b)):
            assert_close(x, y, f"{where}/{i}")
    elif isinstance(a, torch.Tensor):
        assert a.shape == b.shape and a.dtype == b.dtype, (where, a.shape, b.shape, a.dtype, b.dtype)
        assert torch.allclose(a.double(), b.double(), rtol=1e-4, atol=1e-6), (where, float((a.double() - b.double()).abs().max()))
    elif isinstance(a, float):
        assert abs(a - b) <= 1e-6 * max(1.0, abs(a)), (where, a, b)
    else:
        assert a == b, (where, a, b)


def find_free_port():
    with socket.socket(socket.AF_INET, socket.SOCK_STREAM) as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, fn, args, ret):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port), INTERNEVO_FORCE_DIST="1")
    try:
        import torch

        torch.set_num_threads(1)   # several ranks share the cores of one box: intra-op threading only adds contention
        out = fn(rank, world, *args)
        ret[rank] = ("ok", out)
    except Exception:
        ret[rank] = ("err", traceback.format_exc())
    finally:
        try:
            from internevo_b200.core.context import global_context as gpc

            gpc.destroy()
        except Exception:
            pass


def run_distributed(fn, world, *args, timeout=300):
    """Run ``fn(rank, world, *args)`` in ``world`` processes; returns the list of results, raises on any failure.  A
    rendezvous port that another process grabbed between ``find_free_port`` and the bind is retried on a fresh port."""
    for attempt in range(3):
        try:
            return _run_distributed_once(fn, world, *args, timeout=timeout)
        except AssertionError as e:
            if "EADDRINUSE" not in str(e) or attempt == 2:
                raise


def _run_distributed_once(fn, world, *args, timeout=300):
    ctx = mp.get_context("spawn")
    mgr = ctx.Manager()
    ret = mgr.dict()
    port = find_free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, fn, args, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout)
    for p in procs:
        if p.is_alive():
            p.terminate()
            raise TimeoutError("distributed test timed out")
    errs = [f"rank {r}: {v[1]}" for r, v in sorted(ret.items()) if v[0] == "err"]
    assert not errs, "\n".join(errs)
    assert len(ret) == world, f"only {len(ret)} of {world} ranks reported"
    return [ret[r][1] for r in range(world)]


def tiny_config(tp=1, pp=1, zero1=-1, mode="mtp", dtype="torch.float32", num_layers=4, micro_num=2, num_chunks=1,
                model_type="INTERNLM2_PUBLIC", wp=1, hidden=64, heads=4, kv_heads=2, seq_len=32, micro_bsz=2,
                vocab=128, checkpoint=False, fsdp=False, **model_extra):
    model = dict(checkpoint=checkpoint, num_chunks=num_chunks, num_attention_heads=heads, embed_split_hidden=True,
                 vocab_size=vocab, embed_grad_scale=1, parallel_output=True, hidden_size=hidden, num_layers=num_layers,
                 mlp_ratio=2, apply_post_layer_norm=False, dtype=dtype, norm_type="rmsnorm",
                 layer_norm_epsilon=1e-5, use_flash_attn=True)
    if model_type != "INTERNLM" and "MoE" not in model_type:
        model.update(no_bias=True, num_kv_attention_heads=kv_heads)
    model.update(model_extra)
    return dict(
        JOB_NAME="test", model_type=model_type, ckpt=dict(enable_save_ckpt=False, auto_resume=False),
        data=dict(seq_len=seq_len, micro_num=micro_num, micro_bsz=micro_bsz, valid_every=0, pack_sample_into_one=False,
                  total_steps=10, skip_batches="", rampup_batch_size="", min_length=0, train_folder=None,
                  valid_folder=None, num_random_samples=600),
        grad_scaler=dict(fp16=dict(initial_scale=2**10, min_scale=1, growth_interval=1000), growth_factor=2,
                         backoff_factor=0.5, max_scale=2**24, hysteresis=2),
        hybrid_zero_optimizer=dict(overlap_sync_grad=False, overlap_sync_param=False, clip_grad_norm=1.0),
        loss=dict(label_smoothing=0),
        adam=dict(lr=1e-3, adam_beta1=0.9, adam_beta2=0.95, adam_beta2_c=0, adam_eps=1e-8, weight_decay=0.01),
        lr_scheduler=dict(total_steps=10, init_steps=0, warmup_ratio=0.1, eta_min=1e-4, last_epoch=-1),
        beta2_scheduler=dict(init_beta2=0.95, c=0, cur_iter=-1),
        model=model, enable_tb=False,
        parallel=dict(zero1=dict(size=zero1, fsdp=fsdp), tensor=dict(size=tp, mode=mode),
                      pipeline=dict(size=pp, interleaved_overlap=True), weight=dict(size=wp, overlap=True, memory_pool=True)),
    )


def build_trainer(config, seed=1024):
    """launch + model + optimizer + trainer through the public API; returns (trainer, optimizer, model, criterion)."""
    import internevo_b200 as fw
    from internevo_b200.initialize import initialize_distributed_env
    from internevo_b200.models.losses import FlashGPTLMLoss
    from internevo_b200.train import get_scheduler_hooks, initialize_isp_communicator, initialize_model, initialize_optimizer

    initialize_distributed_env(config=config, launcher="torch", seed=seed)
    model = initialize_model()
    isp = initialize_isp_communicator(model)
    crit = FlashGPTLMLoss(parallel_output=True, label_smoothing=0)
    opt, b2, lrs = initialize_optimizer(model, isp)
    trainer, _, _, _ = fw.initialize_trainer(model=model, optimizer=opt, criterion=crit, lr_scheduler=lrs,
                                             beta2_scheduler=b2, scheduler_hooks=get_scheduler_hooks(None, opt, isp))
    trainer.train()
    return trainer, opt, model, crit


def synthetic_batch(micro_num, T, vocab, seed=0, segments=2):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(1, vocab, (micro_num, T), generator=g)
    labels = torch.cat([ids[:, 1:], torch.full((micro_num, 1), -100, dtype=torch.long)], 1)
    seg = T // segments
    cu = torch.tensor([[i * seg for i in range(segments)] + [T]] * micro_num, dtype=torch.int32)
    labels[:, seg - 1:: seg] = -100
    idx = torch.cat([torch.arange(seg)] * segments + [torch.arange(T - seg * segments)]).repeat(micro_num, 1)
    return {"input_ids": ids, "cu_seqlens": cu, "indexes": idx}, labels
