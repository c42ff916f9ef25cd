"""``args_sanity_check`` on one of the reference's OWN config files, run against the reference and against this repository
(``internlm`` alias); prints the resulting configuration (see ``test_reference_differential_cpu.py``).  A ``.json`` config holds
the values a config file defines, as ``Config.from_file`` loaded them.

    python differential_config_probe.py <root that provides `internlm`> <config file or .json> <output json>
"""
import json
import sys

root, cfgfile, dst = sys.argv[1], sys.argv[2], sys.argv[3]
sys.path.insert(0, root)

from internlm.core.context import ParallelMode  # noqa: E402
from internlm.core.context import global_context as gpc  # noqa: E402
from internlm.core.context.parallel_context import Config  # noqa: E402

gpc._config = Config(json.load(open(cfgfile))) if cfgfile.endswith(".json") else Config.from_file(cfgfile)
gpc.is_rank_for_log = lambda: False
gpc.get_world_size = lambda mode: 8 if mode in (ParallelMode.GLOBAL, ParallelMode.DATA) else 1   # an 8-GPU data-parallel job
gpc.is_initialized = lambda mode: True

from internlm.initialize.launch import args_sanity_check  # noqa: E402

args_sanity_check()


def plain(x):
    if isinstance(x, dict):
        return {str(k): plain(v) for k, v in sorted(x.items(), key=lambda kv: str(kv[0]))}
    if isinstance(x, (list, tuple)):
        return [plain(v) for v in x]
    if isinstance(x, (int, float, str, bool)) or x is None:
        return x
    return repr(x)


json.dump(plain(dict(gpc._config)), open(dst, "w"))
print("PROBE_OK")
