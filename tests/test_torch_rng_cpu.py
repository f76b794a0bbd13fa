"""The torch-stream extension ("rng_stream": "torch") without a GPU: the host advance formula, the config key, the
shard rejection and the ctypes layouts."""
import ctypes

import pytest


def _advance(n, sms, tps):
    """calc_execution_policy of ATen/native/cuda/DistributionTemplates.h: grid of min(SMs x tps / 256, ceil(n / 256))
    blocks of 256 threads, 4 elements per thread and round, 4 offsets per round."""
    if n == 0:
        return 0
    g = min(sms * (tps // 256), (n + 255) // 256)
    return ((n - 1) // (256 * g * 4) + 1) * 4


@pytest.mark.parametrize("sms, tps", [(148, 2048), (132, 2048), (1, 256)])
def test_advance_matches_formula_across_regime_edges(sms, tps):
    from leibnizgym_b200 import _native
    lib = _native.load()
    T = 256 * sms * (tps // 256)
    sizes = {0, 1, 3, 4, 255, 256, 257, 4099, 16384, 18 * 16384, T - 1, T, T + 1, 4 * T - 1, 4 * T, 4 * T + 1,
             8 * T, 8 * T + 1, 18 * 65536, 1212416, 1212417, 18 * 262144, 18 * (1 << 23)}
    for n in sorted(sizes):
        assert lib.lg_torch_philox_advance(n, sms, tps) == _advance(n, sms, tps), n
    assert lib.lg_torch_philox_advance(10, 0, 2048) == 0   # no device geometry: nothing to say


def test_rng_stream_key():
    from leibnizgym_b200.config import resolve_config
    from leibnizgym_b200.params import build_params
    from leibnizgym_b200 import _native
    cfg = resolve_config({"command_mode": "torque"})
    assert cfg["rng_stream"] == "philox"
    assert build_params(cfg, 8).rng_stream == _native.RNG_STREAMS["philox"] == 0
    cfg["rng_stream"] = "torch"
    p = build_params(cfg, 8, sm_count=148, threads_per_sm=2048)
    assert (p.rng_stream, p.sm_count, p.threads_per_sm) == (1, 148, 2048)
    for bad in ("Torch", "cpu", None, 1):
        cfg["rng_stream"] = bad
        with pytest.raises(ValueError):
            build_params(cfg, 8)


def test_torch_stream_rejects_sharding():
    from leibnizgym_b200.env import TrifingerEnv
    with pytest.raises(ValueError, match="world_size"):
        TrifingerEnv({"command_mode": "torque", "num_instances": 8, "rng_stream": "torch"}, rank=0, world_size=2,
                     verbose=False)


def test_ctypes_layouts():
    from leibnizgym_b200 import _native
    lib = _native.load()
    assert lib.lg_struct_size(6) == ctypes.sizeof(_native.LgTorchRng) == 48
    assert _native.LgTorchRng.offset.offset == 8
    assert _native.LgBuffers.torch_rng.offset == ctypes.sizeof(_native.LgBuffers) - 8
    assert _native.LgParams.stats_num_envs.offset + 8 <= 168   # the hot block is unchanged
    assert lib.lg_struct_size(0) == ctypes.sizeof(_native.LgParams)
    assert lib.lg_torch_philox(0, 2, 4, 0, None, None) == -1   # offsets are multiples of 4
