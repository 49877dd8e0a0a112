"""Drop-in proof: the SAME reference-signature calls (nn::gptq::gptq_gemm_k_major, nn::multi_query_attention_rag_buffer,
nn::LayerNorm, int8_op::*, nn::fp8::dynamic_scaled_quant ... driven by oracle/ref_shim.cu over every case of
oracle/golden_cases.py) are executed twice on the B200:

  * oracle/_ref/libzl_ref.so     -- the reference's own kernels,
  * oracle/_ref/libzl_dropin.so  -- integration/zl_nn_dropin.cpp, i.e. OUR definitions of those symbols on top of
                                    libzhilight_b200.so (none of the reference's hot-path kernel files is linked),

each in its own process, and the outputs are compared: integer / index work bit-exact, fp16 within the tolerances of
north_star (1e-3 rel; 2e-3 where the reference itself accumulates 8 products in fp16).  Skipped when the two
libraries were not built (they need /root/reference at build time; the built files travel to the GPU box)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.helpers import rel_l2

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref", "libzl_ref.so")
DROPIN = os.path.join(ROOT, "oracle", "_ref", "libzl_dropin.so")

# float outputs: (file, key prefix) -> tolerance; everything not listed that is floating point uses 1e-3
FLOAT_TOL = {"ref_gemv_asym": 2e-3, "ref_gemv_sym": 2e-3, "ref_gate_in": 2e-3, "ref_kv8": 3e-3}
BF16_KEYS = ("_bf16",)


def _generate(out_dir, lib):
    r = subprocess.run([sys.executable, "-m", "oracle.gen_ref_golden", out_dir, lib], cwd=ROOT, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_reference_signature_calls_agree(lib, cuda, tmp_path):
    if not (os.path.exists(REF) and os.path.exists(DROPIN)):
        pytest.skip("oracle/_ref/libzl_ref.so / libzl_dropin.so not built")
    a, b = str(tmp_path / "ref"), str(tmp_path / "dropin")
    _generate(a, REF)
    _generate(b, DROPIN)
    files_ref = sorted(f for f in os.listdir(a) if f.endswith(".npz"))
    files = sorted(f for f in os.listdir(b) if f.endswith(".npz"))
    # the drop-in library has no Marlin (QuantType 8 is served by the GPTQ kernels): every other golden case is produced by both
    assert len(files) >= 13 and set(files) <= set(files_ref) and set(files_ref) - set(files) <= {"ref_marlin.npz"}
    checked = 0
    for f in files:
        name = f[:-4]
        with np.load(os.path.join(a, f)) as ga, np.load(os.path.join(b, f)) as gb:
            assert sorted(ga.files) == sorted(gb.files), f
            for k in ga.files:
                x, y = ga[k], gb[k]
                assert x.shape == y.shape, (f, k)
                if x.dtype.kind == "U" or np.issubdtype(x.dtype, np.integer) or \
                        k in ("sx_f16", "sx_bf16", "f8_s_f16", "f8_s_bf16", "s"):        # "U": digests of large outputs
                    np.testing.assert_array_equal(x, y, err_msg="%s:%s" % (f, k))      # integer / scale work: bit-exact
                else:
                    tol = FLOAT_TOL.get(name, 1e-3)
                    if k.endswith(BF16_KEYS):
                        tol = max(tol, 4e-3)
                    if name == "ref_int8" and k == "allreduce":
                        # int8-g32 payload: both sides within one quantisation step of each other
                        step = np.abs(x.astype(np.float32)).max() / 127.0
                        np.testing.assert_allclose(x.astype(np.float32), y.astype(np.float32), atol=1.01 * step)
                    else:
                        err = rel_l2(y.astype(np.float32), x.astype(np.float32))
                        assert err <= tol, "%s:%s rel %.3e > %.1e" % (f, k, err, tol)
                checked += 1
    assert checked >= 40
