"""The reference's own CLI (src/main.cpp, UNMODIFIED, with the nnet_data.cpp the reference's own exporter writes for
synth_state_dict(0)), run by tests/golden/make_golden.py: on e2e.npz's input (digests in reference_digests.json) and
on 60 synthetic hops (cli.npz, its PCM file and feature_test.raw).  The drop-in library librnnoise_b200.so, driven
through the rnnoise.h calls and frame loop of src/main.cpp, must give the same PCM file within +-1 LSB and the same
feature_test.raw (g, r) within 1e-4."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN
from util import digest, reference_digests


def test_reference_cli_matches_golden_and_oracle(oracle, model0):
    """CPU: the true reference binary == the golden fixture (made through the harness) == the oracle."""
    g = np.load(os.path.join(GOLDEN, "e2e.npz"))
    want = reference_digests()["cli"]
    assert digest(g["cli_out16"]) == want["e2e_out16"] and digest(g["cli_gr"]) == want["e2e_gr"]
    o16, ogr = oracle.run_pcm16(model0, g["x16"])
    assert np.array_equal(o16, g["cli_out16"]) and np.array_equal(ogr.view(np.int32), g["cli_gr"].view(np.int32))


def _run_shim_like_cli(x16, model, feature_path):
    """src/main.cpp's loop on librnnoise_b200.so: int16 / 32768 -> rnnoise_process_frame in place, g/r appended to
    a FILE* -> * 32768 -> int16, the first hop dropped."""
    from percepnet_b200 import build
    libc = C.CDLL(None)
    libc.fopen.restype = C.c_void_p
    libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
    libc.fclose.argtypes = [C.c_void_p]
    shim = C.CDLL(build.SHIM)
    create = shim._Z14rnnoise_createP8RNNModel
    create.restype, create.argtypes = C.c_void_p, [C.c_void_p]
    process = shim._Z21rnnoise_process_frameP12DenoiseStatePfPKfP8_IO_FILE
    process.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    destroy = shim._Z15rnnoise_destroyP12DenoiseState
    destroy.argtypes = [C.c_void_p]
    m = model.as_c_model()
    st = create(C.addressof(m))
    assert st, "rnnoise_create failed"
    f = libc.fopen(feature_path.encode(), b"wb")
    x = np.empty(480, np.float32)
    out = []
    for t in range(x16.size // 480):
        x[:] = x16[480 * t:480 * (t + 1)].astype(np.float32) / np.float32(32768)
        process(st, x.ctypes.data, x.ctypes.data, f)
        if t:
            out.append((x * np.float32(32768)).astype(np.int32).astype(np.int16))
    destroy(st)
    libc.fclose(f)
    return np.concatenate(out), np.fromfile(feature_path, dtype=np.float32).reshape(-1, 68)


@pytest.mark.gpu
def test_dropin_cli_on_gpu(tmp_path, model0):
    from percepnet_b200.synth import synth_pcm, to_int16
    x16 = to_int16(synth_pcm(1, 60, seed=2024)[0])
    g = np.load(os.path.join(GOLDEN, "cli.npz"))
    ref_out, ref_gr = g["out16"], g["gr"]
    for nn in ("fp32", "tensor"):                                    # PNB_SHIM_NN selects the shim's network path
        os.environ["PNB_SHIM_NN"] = nn
        try:
            out, gr = _run_shim_like_cli(x16, model0, str(tmp_path / f"feature_{nn}.raw"))
        finally:
            del os.environ["PNB_SHIM_NN"]
        assert out.shape == ref_out.shape == ((60 - 1) * 480,)      # first hop dropped, src/main.cpp:37-38
        assert np.abs(out.astype(np.int32) - ref_out.astype(np.int32)).max() <= 1, nn
        assert gr.shape == ref_gr.shape == (60, 68)
        rel = np.abs(gr - ref_gr) / np.maximum(np.abs(ref_gr), 1e-6)
        assert rel.max() < 1e-4, nn
