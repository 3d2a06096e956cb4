"""CPU: the C-ABI library builds, loads, and exports every symbol include/librec_b200.h declares."""
import ctypes
import os
import re

import pytest

from conftest import ROOT


def _declared():
    src = open(os.path.join(ROOT, "include", "librec_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lrk_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_are_exported(capi):
    names = _declared()
    assert len(names) >= 20
    lib = ctypes.CDLL(capi.lib_path())
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    # and the ctypes binding knows every one of them
    assert sorted(capi.SIGNATURES) == names


def test_version_and_abi(capi):
    L = capi.load()
    assert b"sm_100a" in L.lrk_version()
    assert L.lrk_abi_version() == 1
    assert L.lrk_device_count() >= 0


def test_no_cpu_fallback(capi):
    """without a B200 every compute entry fails loudly -- there is no CPU path in the product.  The check runs in a child process
    that sees no CUDA device, so that it also runs on a machine that has one."""
    import subprocess
    import sys
    child = ("import sys\nsys.path.insert(0, %r)\nfrom librec_b200 import capi\nassert capi.device_count() == 0\n"
             "try:\n    capi.Handle(capi.MODEL_BIASEDMF, 8)\nexcept capi.LibrecException as e:\n    print('status', e.status)\n") % ROOT
    r = subprocess.run([sys.executable, "-c", child], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr
    status = re.findall(r"^status (-?\d+)$", r.stdout, flags=re.M)
    assert len(status) == 1 and int(status[0]) in (capi.ERR_CUDA, capi.ERR_INVALID), r.stdout


def test_bad_config_is_rejected(capi):
    for kw in (dict(model=9, num_factors=8), dict(model=0, num_factors=0), dict(model=0, num_factors=257)):
        with pytest.raises(capi.LibrecException):
            capi.Handle(kw["model"], kw["num_factors"])


def test_product_never_imports_oracle():
    """librec_b200/ must not reference oracle/ (the oracle is test infrastructure)"""
    bad = []
    for dp, _, fs in os.walk(os.path.join(ROOT, "librec_b200")):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".inc", ".cpp", ".hpp", ".h")):
                txt = open(os.path.join(dp, f), errors="ignore").read()
                if re.search(r"(from|import)\s+oracle|lrk_oracle|lro_", txt):
                    bad.append(f)
    assert not bad, bad


def test_enum_values_agree_across_header_binding_and_java_shim(capi):
    """the integer constants of include/librec_b200.h, librec_b200/capi.py and java/.../LibrecB200.java must not drift apart"""
    src = open(os.path.join(ROOT, "include", "librec_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    header = {m.group(1): int(m.group(2)) for m in re.finditer(r"\b(LRK_[A-Z_]+)\s*=\s*(-?\d+)", src)}
    for name in ("MODEL_BIASEDMF", "MODEL_PMF", "MODEL_BPR", "MODEL_RANKSGD", "MODEL_GBPR", "MODEL_SVDPP", "MODEL_AOBPR", "MODEL_WRMF", "MODEL_EALS", "UPDATE_ATOMIC", "UPDATE_HOGWILD",
                 "UPDATE_REFERENCE_ORDER", "OK", "ERR_INVALID", "ERR_CUDA", "ERR_NCCL", "ERR_NOMEM", "ERR_DIVERGED"):
        assert getattr(capi, name) == header["LRK_" + name], name
    java = open(os.path.join(ROOT, "java", "net", "librec", "recommender", "cuda", "LibrecB200.java")).read()
    jconst = {m.group(1): int(m.group(2)) for m in re.finditer(r"\b(MODEL_[A-Z]+)\s*=\s*(\d+)", java)}
    for name, value in jconst.items():
        assert header["LRK_" + name] == value, name
    assert set(jconst) == {"MODEL_BIASEDMF", "MODEL_PMF", "MODEL_BPR", "MODEL_RANKSGD", "MODEL_GBPR", "MODEL_SVDPP", "MODEL_AOBPR", "MODEL_WRMF", "MODEL_EALS"}
    # the bad-model guard of test_bad_config_is_rejected relies on 9 being out of range
    assert max(v for k, v in header.items() if k.startswith("LRK_MODEL_")) < 9


def test_jni_forwarder_compiles_and_covers_every_export():
    """java/librec_b200_jni.c is the reference-side JNI binding of the C ABI.  No JDK in this image: it is compiled against a
    minimal stand-in for jni.h (tests/stubs/jni.h) with -Wall -Werror, every lrk_* export must be forwarded by it, and every
    JNI function must have a `static native` declaration of the same name in LibrecB200.java (and vice versa)."""
    import shutil
    import subprocess
    src = os.path.join(ROOT, "java", "librec_b200_jni.c")
    gcc = shutil.which("gcc")
    assert gcc, "gcc missing"
    r = subprocess.run([gcc, "-fsyntax-only", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "tests", "stubs"),
                        "-I", os.path.join(ROOT, "include"), src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    code = re.sub(r"/\*.*?\*/", "", open(src).read(), flags=re.S)
    called = set(re.findall(r"\b(lrk_[a-z0-9_]+)\s*\(", code))
    assert sorted(called) == _declared()
    jni_names = set(re.findall(r"LRK_JNI\((\w+)\)", code)) - {"name"}      # "name" is the macro parameter
    java = open(os.path.join(ROOT, "java", "net", "librec", "recommender", "cuda", "LibrecB200.java")).read()
    natives = set(re.findall(r"static native [\w\[\]]+ (\w+)\(", java))
    assert jni_names == natives, (jni_names ^ natives)


def test_every_model_has_a_java_shim_class():
    """each MODEL_* of LibrecB200.java is returned by the model() of exactly one *CudaRecommender.java (what rec.recommender.class names)"""
    jdir = os.path.join(ROOT, "java", "net", "librec", "recommender", "cuda")
    consts = set(re.findall(r"\b(MODEL_[A-Z]+)\s*=", open(os.path.join(jdir, "LibrecB200.java")).read()))
    used = {}
    for f in sorted(os.listdir(jdir)):
        if f.endswith("CudaRecommender.java"):
            for m in re.findall(r"int model\(\)\s*\{\s*return LibrecB200\.(MODEL_[A-Z]+);", open(os.path.join(jdir, f)).read()):
                used.setdefault(m, []).append(f)
    assert set(used) == consts, (sorted(consts - set(used)), sorted(set(used) - consts))
    assert all(len(v) == 1 for v in used.values()), used
