"""A fixed slice of tools/fuzz_module_configs.py in the CPU tier: random user module configs as TEXT through the reference's
own shaders (interpreter; recorded where the reference tree is absent), through config reader + oracle, and through config
reader + product arithmetic.  The reader falls back to the package's own config directory, not the reference's."""
import importlib.util
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SHADERS = "/root/reference/shaders/glava"
OWN_CONFIG = os.path.join(ROOT, "glava_b200", "config")


@pytest.fixture(scope="module")
def fuzz(built):
    spec = importlib.util.spec_from_file_location("fuzz_module_configs", os.path.join(ROOT, "tools", "fuzz_module_configs.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


# 207 / 267: circle, C_SMOOTH 0, non-native opacity (the pass-through stage 2); 131: a 1-LSB radial pixel; 5 / 12 / 26 / 33:
# setsmoothpass flipped in rc.glsl and / or a random smooth_parameters.glsl (the three consistent / stale-header variants of
# tools/fuzz_module_configs.py); 166 / 586 / 803 / 985:
# the same with a smooth factor whose "%.6f" header literal differs from the request's float; the rest: a spread
@pytest.mark.parametrize("seed", [207, 267, 131, 5, 12, 26, 33, 166, 586, 803, 985] + list(range(40, 66)))
def test_random_module_config(fuzz, ref_record, seed):
    module = ["bars", "radial", "circle", "graph", "wave"][seed % 5]
    w, h = [(40, 28), (41, 27), (38, 30)][seed % 3]

    def frame(d, *args):
        return ref_record.call("shader_frame", lambda *a: fuzz.shader_frame(d, *a[1:]), (d,) + args, whole=True)
    text, want, oracle, product = fuzz.run(seed, module, w, h, native=(seed % 4 != 3), config_tail=OWN_CONFIG, frame=frame,
                                           smooth_in_shader=((1 + seed // 7 % 3) if (seed % 7 == 5 and module in ("bars", "radial", "circle", "graph")) else False))
    assert want.any(), text
    assert np.array_equal(oracle, want), (seed, module, text)
    assert int(np.abs(product.astype(int) - want.astype(int)).max()) <= 1, (seed, module, text)
    assert (product != want).any(axis=2).sum() <= 0.005 * w * h, (seed, module, text)
