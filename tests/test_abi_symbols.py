"""The C-ABI library builds for sm_100a on a CPU-only box, loads, and exports every function that
include/rtgs_b200.h declares (no compute calls here — those are the `gpu` tests)."""
import ctypes
import re
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def _declared():
    text = (ROOT / "include" / "rtgs_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rtgs_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_the_path():
    names = _declared()
    for must in ("rtgs_scene_create", "rtgs_scene_build_bvh", "rtgs_render", "rtgs_render_host",
                 "rtgs_trace_closest", "rtgs_generate_rays", "rtgs_scene_read_lbvh", "rtgs_scene_destroy"):
        assert must in names


def test_library_exports_every_declared_symbol(lib):
    from rtgs import _native
    names = _declared()
    raw = ctypes.CDLL(str(_native.LIB_PATH))
    for n in names:
        assert hasattr(raw, n), f"{n} declared in include/rtgs_b200.h but not exported"
    assert sorted(_native.SIGNATURES) == names, "ctypes SIGNATURES out of sync with the header"
    assert lib.rtgs_abi_version() == 3


def test_struct_and_enum_mirrors_match_the_header():
    """The ctypes mirrors in rtgs/_native.py are written by hand: field names and order of rtgs_render_stats (every
    field uint64_t), and the option numbers, must be those of the header - a drifted mirror corrupts memory silently."""
    from rtgs import _native
    text = (ROOT / "include" / "rtgs_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    body = re.search(r"typedef struct rtgs_render_stats \{(.*?)\} rtgs_render_stats;", text, flags=re.S).group(1)
    decls = [d.strip() for d in body.split(";") if d.strip()]
    assert all(d.startswith("uint64_t ") for d in decls)
    assert [d.split()[1] for d in decls] == [n for n, _ in _native.rtgs_render_stats._fields_]
    assert ctypes.sizeof(_native.rtgs_render_stats) == 8 * len(decls)
    enum = dict(re.findall(r"\b(RTGS_OPT_[A-Z_]+)\s*=\s*(\d+)", text))
    for name, value in enum.items():
        assert getattr(_native, name[len("RTGS_"):]) == int(value), name


def test_errors_are_reported_not_thrown(lib):
    # argument validation happens before any CUDA call, so this is safe without a GPU
    out = ctypes.c_void_p()
    st = lib.rtgs_scene_create(0, 0, None, None, None, None, None, None, ctypes.byref(out))
    assert st == -1 and b"invalid argument" in lib.rtgs_last_error()
    assert lib.rtgs_render(None, None, 0, 0, 1, 1, 16, 0.0, 0, 0, None, None, None, None) == -1


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    # monkeypatch restores the module afterwards; reloading it instead would replace the ctypes classes
    # (rtgs_camera, ...) that the already loaded library's argtypes name, and break every later render call
    from rtgs import _native
    monkeypatch.setattr(_native, "_lib", None)
    monkeypatch.setattr(_native, "LIB_PATH", tmp_path / "nope.so")
    try:
        _native.load()
    except ImportError as e:
        assert "no CPU fallback" in str(e)
    else:
        raise AssertionError("loading a missing library must raise")
