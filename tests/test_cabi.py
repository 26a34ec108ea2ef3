"""The C-ABI library loads on a CPU-only box and exports every symbol that
include/b200vlm.h declares (no compute calls here)."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "b200vlm.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", src)))


def test_library_builds_and_exports_every_declared_symbol():
    from mlx_vlm_b200.build import build
    from mlx_vlm_b200 import _native as N
    build()
    lib = N.lib()
    names = _declared()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/b200vlm.h but not exported"
        assert n in N.SIGNATURES, f"{n} has no ctypes signature in _native.py"
    assert set(N.SIGNATURES) <= set(names), sorted(set(N.SIGNATURES) - set(names))
    assert lib.b200_abi_version() == 1
    assert isinstance(lib.b200_last_error(), bytes)


def test_ctypes_signatures_match_the_header():
    """every declaration of include/b200vlm.h and its ctypes signature in _native.py take the same number of arguments
    (a drifted binding would pass garbage through the C ABI without any error)"""
    import ctypes as C
    from mlx_vlm_b200 import _native as N
    src = open(os.path.join(ROOT, "include", "b200vlm.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"//[^\n]*", "", src)
    decls = re.findall(r"\b(b200_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", src, flags=re.S)
    assert len(decls) >= 60
    seen = set()
    for name, args in decls:
        args = " ".join(args.split())
        n = 0 if args in ("", "void") else args.count(",") + 1
        assert name in N.SIGNATURES, name
        sig = N.SIGNATURES[name][1]
        assert len(sig) == n, f"{name}: header has {n} arguments, _native.py {len(sig)}"
        for i, (decl, ct) in enumerate(zip(args.split(",") if n else [], sig)):   # and the same kind, argument by argument
            decl = decl.strip()
            kind = "ptr" if "*" in decl else " ".join(decl.split()[:-1])
            want = {"ptr": None, "int": C.c_int, "unsigned": C.c_uint, "long": C.c_long, "float": C.c_float}[kind]
            if want is None:
                assert ct in (C.c_void_p, C.c_char_p) or issubclass(ct, C._Pointer), f"{name} arg {i}: `{decl}` bound as {ct}"
            else:
                assert ct is want, f"{name} arg {i}: `{decl}` bound as {ct}"
        seen.add(name)
    assert seen == set(N.SIGNATURES), sorted(set(N.SIGNATURES) ^ seen)


def test_no_oracle_import_in_product():
    """the product path may not import or execute anything under oracle/"""
    pkg = os.path.join(ROOT, "mlx_vlm_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                txt = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), os.path.join(dp, f)


def test_engine_refuses_without_gpu():
    """a model placed on the CPU gets no engine, whether or not the machine has a GPU"""
    import pytest
    from mlx_vlm_b200 import _native as N
    from mlx_vlm_b200.models.qwen2_vl import Model
    from mlx_vlm_b200.models.qwen2_vl.config import qwen2_vl_2b_config
    m = Model(qwen2_vl_2b_config(), device="cpu")
    with pytest.raises(N.B200Error):
        m.engine  # no CPU fallback: fails loudly
