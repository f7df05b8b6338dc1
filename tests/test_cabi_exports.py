"""CPU tests of the drop-in boundary: the C-ABI library builds, loads and exports every symbol
include/describealign_b200.h declares; without a CUDA device the product path fails loudly
(no CPU fallback); the host-side mirror has the reference's names and signatures.
No compute is launched here.
"""
import ctypes
import inspect
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "describealign_b200.h")


@pytest.fixture(scope="module")
def lib():
    from describealign_b200 import _cabi, build
    build.build()
    return _cabi.load()


def _declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dab_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported(lib):
    names = _declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in the header but not exported"


def test_binding_covers_header():
    from describealign_b200 import _cabi
    assert sorted(_cabi.EXPORTS) == _declared_symbols()


def test_abi_version_and_struct_layout(lib):
    from describealign_b200 import _cabi
    assert lib.dab_abi_version() == 2
    assert ctypes.sizeof(_cabi.Corridor) == 32       # 4 x int32 + 2 x double
    assert ctypes.sizeof(_cabi.StageBIn) == 56       # 6 x float, 2 x int64, int32 + padding, pointer
    assert ctypes.sizeof(_cabi.Stats) == 15 * 8


def test_no_cpu_fallback(lib):
    """On a box without a GPU the context cannot be created and every API entry raises."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    from describealign_b200 import _cabi, api
    h = ctypes.c_void_p()
    assert lib.dab_create(-1, ctypes.byref(h)) != 0
    assert b"no CPU fallback" in lib.dab_last_error(None)
    with pytest.raises(_cabi.DabError):
        api.get_energy(np.zeros((1, 4410), np.float16))
    with pytest.raises(_cabi.DabError):
        api.align_pcm(np.zeros((4410, 1), np.int16), np.zeros((4410, 1), np.int16))


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from describealign_b200 import _cabi
    monkeypatch.setattr(_cabi, "_lib", None)
    monkeypatch.setattr(_cabi, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_cabi.DabError, match="no CPU fallback"):
        _cabi.load()


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure: nothing under describealign_b200/ may reference it."""
    pkg = os.path.join(ROOT, "describealign_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "liboracle" not in src, f


def test_mirror_has_reference_signatures():
    """describealign.py:545, 557, 575, 595: same names and positional parameters."""
    from describealign_b200 import api
    assert list(inspect.signature(api.get_energy).parameters) == ["arr"]
    assert list(inspect.signature(api.get_zero_crossings).parameters) == ["arr"]
    assert list(inspect.signature(api.get_freq_bands).parameters) == ["arr"]
    assert list(inspect.signature(api.align).parameters)[:4] == [
        "video_features", "audio_desc_features", "video_energy", "audio_desc_energy"]


def test_launcher_patches_a_module():
    import types
    from describealign_b200 import api, launcher
    fake = types.ModuleType("describealign")
    for n in ("get_energy", "get_zero_crossings", "get_freq_bands", "align"):
        setattr(fake, n, lambda *a, **k: None)
    launcher.patch(fake)
    assert fake.align is api.align and fake.get_freq_bands is api.get_freq_bands
    assert callable(fake._reference_align)
    broken = types.ModuleType("describealign")
    with pytest.raises(AttributeError):
        launcher.patch(broken)


def test_launcher_optional_patches(monkeypatch):
    """replace_aligned_segments is patched where the module has it; parse_audio_from_file only on request, and its
    replacement hands mono tracks over as DevicePcm and stereo tracks as host arrays with remembered features."""
    import types
    import numpy as np
    from describealign_b200 import api, decode, launcher, stretch
    fake = types.ModuleType("describealign")
    for n in ("get_energy", "get_zero_crossings", "get_freq_bands", "align", "replace_aligned_segments", "parse_audio_from_file"):
        setattr(fake, n, lambda *a, **k: None)
    fake.get_ffmpeg = lambda: "/opt/ffmpeg"
    original_parse = fake.parse_audio_from_file
    launcher.patch(fake)
    assert fake.replace_aligned_segments is stretch.replace_aligned_segments
    assert fake.parse_audio_from_file is original_parse          # untouched without decode=True
    launcher.patch(fake, decode=True)
    assert fake.parse_audio_from_file is not original_parse and fake._reference_parse_audio_from_file is original_parse

    calls = []

    class FakePcm:
        def __init__(self, ch):
            self.ch = ch
        def wait(self):
            return self
        def to_host(self):
            return np.zeros((self.ch, 8), np.float16)
        def features(self):
            return ["e", "z", "b0", "b1", "b2"]
        def close(self):
            calls.append("closed")

    def fake_parse(media_file, num_channels=2, ffmpeg="ffmpeg", command=None):
        calls.append((media_file, num_channels, ffmpeg))
        return FakePcm(num_channels)

    monkeypatch.setattr(decode, "parse_audio_from_file", fake_parse)
    mono = fake.parse_audio_from_file("a.mkv", 1)
    assert isinstance(mono, FakePcm) and calls[-1] == ("a.mkv", 1, "/opt/ffmpeg")
    stereo = fake.parse_audio_from_file("b.mkv", 2)
    assert isinstance(stereo, np.ndarray) and stereo.shape == (2, 8) and calls[-1] == "closed"
    assert api.track_features(stereo) == ["e", "z", "b0", "b1", "b2"]       # from the cache: no upload, no device needed


def test_host_wait_mode_is_validated(lib):
    lib.dab_set_host_wait.argtypes = [ctypes.c_int, ctypes.c_int]
    lib.dab_set_host_wait.restype = ctypes.c_int
    assert lib.dab_set_host_wait(-1, 7) < 0          # unknown mode
    # without a device the call reports the CUDA failure instead of pretending
    from describealign_b200 import _cabi
    if lib.dab_device_count() == 0:
        assert lib.dab_set_host_wait(-1, 2) < 0
        with pytest.raises(_cabi.DabError):
            _cabi.set_host_wait(-1, 2)


def test_scaled_features_follow_from_six_scalars():
    """host_fit.scale_features against the six scalars of host_fit.feature_gains: the scaled arrays are
    exactly audio / std and video * gain / std in float32 - what dab_pair_stage_b_clusters redoes on the device."""
    from describealign_b200 import host_fit
    rng = np.random.default_rng(5)
    n_v, n_a = 5000, 5600
    video = [rng.standard_normal(n_v + (k == 0)).astype(np.float32) for k in range(5)]
    audio = [rng.standard_normal(n_a + (k == 0)).astype(np.float32) for k in range(5)]
    y = np.sort(rng.integers(0, n_v, 900)); x = np.sort(rng.integers(0, n_a, 900))
    a_s, v_s = host_fit.scale_features(video, audio, x, y)
    g, sd, na, nv = host_fit.feature_gains(video, audio, x, y)
    assert a_s.shape == (n_a, 3) and v_s.shape == (n_v, 3) and (na, nv) == (n_a, n_v)
    assert a_s.dtype == v_s.dtype == np.float32
    assert g.dtype == np.float32 and sd.dtype == np.float32 and g.shape == sd.shape == (3,)
    for k in range(3):
        np.testing.assert_array_equal(a_s[:, k], (audio[k][:n_a] / sd[k]).astype(np.float32))
        np.testing.assert_array_equal(v_s[:, k], ((video[k][:n_v] * g[k]).astype(np.float32) / sd[k]).astype(np.float32))
    # float64 features: the device cannot redo numpy's arithmetic from float32 scalars
    video64 = [f.astype(np.float64) for f in video]
    with pytest.raises(TypeError):
        host_fit.feature_gains(video64, audio, x, y)


def test_worker_threads_use_the_process_device(monkeypatch):
    """api.set_device: contexts created lazily in worker threads (CUDA's current device is per thread and
    starts at 0) must be opened on the process's GPU, e.g. LOCAL_RANK under torchrun."""
    import threading
    from describealign_b200 import _cabi, api
    seen = []

    class FakeContext:
        def __init__(self, device=-1):
            seen.append(device)

    monkeypatch.setattr(_cabi, "Context", FakeContext)
    monkeypatch.setattr(api, "_device", -1)
    t = threading.Thread(target=api.context); t.start(); t.join()
    api.set_device(3)
    t = threading.Thread(target=api.context); t.start(); t.join()
    assert seen == [-1, 3]
