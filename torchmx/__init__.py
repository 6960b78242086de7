"""Drop-in import name: `import torchmx` resolves to the B200-native implementation in
`torchmx_b200`, module by module (`torchmx.mx_tensor`, `torchmx.dtypes`, `torchmx.config`,
`torchmx.env_variables`, `torchmx.utils`, `torchmx.ops`, `torchmx.quant_api`,
`torchmx.layers.mx_linear`, `torchmx.kv_cache`), so code and tests written against the reference run unchanged.
"""
import importlib
import sys

import torchmx_b200 as _impl

_ALIASES = ("dtypes", "env_variables", "config", "utils", "mx_tensor", "ops", "mx_gemm", "attention_ops", "mlp_ops", "quant_api", "layers", "layers.mx_linear", "layers.packed_linear", "layers.mx_llama_attention", "layers.tp_linear", "kv_cache")
for _name in _ALIASES:
    try:
        sys.modules[f"{__name__}.{_name}"] = importlib.import_module(f"torchmx_b200.{_name}")
    except ImportError:  # the attention blocks need `transformers`; everything else does not
        if _name not in ("layers.mx_llama_attention", "kv_cache"):
            raise

from torchmx_b200 import MXTensor, config, dtypes, env_variables, mx_tensor, ops, utils  # noqa: E402,F401
from torchmx_b200 import layers, quant_api  # noqa: E402,F401
