"""A tiny model from one folder of HF remote code (``<folder>/configuration_*.py``, ``modeling_*.py``): ``which = ref`` creates random
weights and saves them, ``which = ours`` loads them (no key may be missing or unexpected); both save the logits of the same input
(see ``test_reference_differential_cpu.py``).

    python differential_hf_probe.py <ref|ours|load> <folder with the remote code> <family: internlm|internlm2> <output prefix>

``which = load``: the class of ``<folder>`` takes the weights of ``<prefix>.hf_weights`` (a converted checkpoint) and scores
``<prefix>.ids``.
"""
import importlib.util
import os
import sys
import types

import torch

which, base, family, prefix = sys.argv[1:5]
pkg = types.ModuleType("remote_code")
pkg.__path__ = [base]
sys.modules["remote_code"] = pkg


def load(name):
    spec = importlib.util.spec_from_file_location(f"remote_code.{name}", os.path.join(base, name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[f"remote_code.{name}"] = mod
    spec.loader.exec_module(mod)
    return mod


cfg_mod, model_mod = load(f"configuration_{family}"), load(f"modeling_{family}")
name = "InternLM2" if family == "internlm2" else "InternLM"
kw = dict(vocab_size=64, hidden_size=32, intermediate_size=int(os.environ.get("PROBE_INTERMEDIATE", "64")), num_hidden_layers=2, num_attention_heads=4,
          max_position_embeddings=64, rms_norm_eps=1e-5, attn_implementation="eager")
if family == "internlm2":
    kw.update(num_key_value_heads=2, bias=False, rope_theta=10000)
if which == "load":        # the converted model's MLP width (the trainer rounds it up to a multiple of 256)
    shapes = {k: v.shape for k, v in torch.load(prefix + ".hf_weights").items()}
    kw["intermediate_size"] = next(v[0] for k, v in shapes.items() if k.endswith("feed_forward.w1.weight") or k.endswith("gate_proj.weight"))
cfg = getattr(cfg_mod, name + "Config")(**kw)
if which in ("ref", "load") and getattr(cfg, "rope_scaling", None) is not None:     # "ref" / "load" run the reference's code
    cfg.rope_scaling = None       # transformers 5 fills in a rope dict the 4.x-era reference code does not understand
if which == "ref" and family == "internlm" and hasattr(cfg, "rotary"):
    pass
torch.manual_seed(0)
model = getattr(model_mod, name + "ForCausalLM")(cfg).float().eval()
if which == "load":
    missing, unexpected = model.load_state_dict(torch.load(prefix + ".hf_weights"), strict=False)
    assert not [k for k in missing if "inv_freq" not in k] and not [k for k in unexpected if "inv_freq" not in k], (missing, unexpected)
elif which == "ref":
    for p in model.parameters():
        if p.dim() == 1:
            p.data.add_(0.1 * torch.randn_like(p))
    torch.save(model.state_dict(), prefix + ".weights")
else:
    missing, unexpected = model.load_state_dict(torch.load(prefix + ".weights"), strict=False)
    missing = [k for k in missing if "inv_freq" not in k]
    unexpected = [k for k in unexpected if "inv_freq" not in k]
    assert not missing and not unexpected, (missing, unexpected)
torch.manual_seed(1)
ids = torch.load(prefix + ".ids") if which == "load" else torch.randint(1, 64, (2, 12))
with torch.no_grad():
    logits = model(input_ids=ids).logits
torch.save(logits.float(), f"{prefix}.{which}.logits")
print("PROBE_OK", tuple(logits.shape), flush=True)
