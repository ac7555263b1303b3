"""CPU check of the 80-bin instance of the log-mel kernel's arithmetic (csrc/logmel.cu, MelLayout<80>): the kernel's
__host__ __device__ phases run serially on the host in its warp / lane structure (tests/csrc/logmel_host_test_n.cu built
with -DLOGMEL_NMEL=80: lanes 0-19 own the bins, up to 14 filter taps), compared with the 80-bin numpy reference, which
tests/test_v2_cpu.py pins to WhisperFeatureExtractor(feature_size=80)."""
import os
import subprocess

import numpy as np
import pytest

import helpers
import helpers_v2 as V

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "oracle", "_ref", "logmel_host_test_80")


@pytest.fixture(scope="module")
def binary():
    if not os.path.exists(BIN):
        import __graft_entry__ as g
        g.build_host_tests()
    if not os.path.exists(BIN):
        pytest.skip("host emulation binary not built (no nvcc)")
    return BIN


@pytest.mark.parametrize("name,clip", [
    ("noise30", lambda: helpers.synth_clip(0)),
    ("mod11", lambda: helpers.synth_clip(2, seconds=11.3, kind="mod")),      # zero tail: the per-clip floor is active
    ("silence", lambda: np.zeros(1000, np.float32)),
])
def test_kernel_phases_on_host_match_oracle_80(binary, tmp_path, name, clip):
    from turbo_whisper_workspace_b200.ops import slaney_mel_filters
    x = clip()
    pcm, fb, out = tmp_path / "pcm.f32", tmp_path / "fb.f32", tmp_path / "out.f32"
    x.astype(np.float32).tofile(pcm)
    slaney_mel_filters(80).astype(np.float32).tofile(fb)
    subprocess.run([binary, str(pcm), str(len(x)), str(fb), str(out)], check=True)
    got = np.fromfile(out, dtype=np.float32).reshape(80, 3000)
    np.testing.assert_allclose(got, V.log_mel(x), rtol=1e-4, atol=1e-4)


def test_80_bin_filterbank_needs_14_taps():
    """The 80-filter slaney bank is wider per filter than the 128-filter one: the kernel's tap bound must cover it."""
    from turbo_whisper_workspace_b200.ops import slaney_mel_filters
    for n, taps in ((80, 14), (128, 9)):
        fb = slaney_mel_filters(n)
        spans = [np.ptp(np.nonzero(fb[:, m])[0]) + 1 for m in range(n) if fb[:, m].any()]
        assert max(spans) == taps
