"""The Python side of the C-ABI formats against include/cygym_b200.h: every constant _capi mirrors has the header's value,
the internal record's plane ids match cyg_core.cuh, and the ctypes structs have the C layouts (sizeof / offsetof as the
host compiler lays the header out)."""
import ast
import ctypes as C
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "cygym_b200.h")
CORE = os.path.join(ROOT, "cygym_b200", "csrc", "cyg_core.cuh")
UNUSED_BY_PYTHON = {"CYG_OK", "CYG_BUSY_MAX"}  # header constants no Python code reads


def _c_constants(path):
    """#define NAME <integer> and enum { NAME = <integer>, ... } of a C header -> {NAME: value}."""
    src = re.sub(r"/\*.*?\*/", "", open(path).read(), flags=re.S)
    out = {n: int(v.strip("()").rstrip("uU"), 0) for n, v in re.findall(r"^#define\s+(\w+)\s+(\(?-?(?:0x)?[0-9A-Fa-f]+u?\)?)\s*$", src, re.M)}
    for body in re.findall(r"\benum\s*\{([^}]*)\}", src):
        out.update({n: int(v, 0) for n, v in re.findall(r"(\w+)\s*=\s*(-?\w+)", body)})
    return out


def test_constants_match_the_header():
    from cygym_b200 import _capi as K
    hdr = {n: v for n, v in _c_constants(HEADER).items() if n.startswith("CYG_")}
    assert len(hdr) > 60 and hdr["CYG_S_EADD"] == 15 and hdr["CYG_E_INVAL"] == -22 and hdr["CYG_CK_VALID"] == 1 << 31
    for n, v in hdr.items():
        if n not in UNUSED_BY_PYTHON:
            assert hasattr(K, n[4:]), f"_capi has no {n[4:]} ({n})"
        if hasattr(K, n[4:]):
            assert getattr(K, n[4:]) == v, f"_capi.{n[4:]} = {getattr(K, n[4:])}, {n} = {v}"
    assert sorted(K.BASE_LINES.values()) == [hdr[f"CYG_BL_{b}"] for b in ("NASH", "NO_DEFENSE", "PRESET", "NO_ATTACK")]
    not_counters = {hdr[f"CYG_S_{s}"] for s in ("EPOCH", "FLAGS", "PREV_X", "LOGS")}
    assert sorted(slot for _, _, slot, _ in K.COUNTERS) == sorted(set(range(hdr["CYG_NSCAL"])) - not_counters)
    # _capi is the only module that defines them
    names = {n[4:] for n in hdr}
    pkg = os.path.join(ROOT, "cygym_b200")
    for f in sorted(os.listdir(pkg)):
        if f.endswith(".py") and f != "_capi.py":
            tree = ast.parse(open(os.path.join(pkg, f)).read())
            defined = {t.id for node in tree.body if isinstance(node, ast.Assign) for tgt in node.targets
                       for t in (tgt.elts if isinstance(tgt, ast.Tuple) else [tgt]) if isinstance(t, ast.Name)}
            assert not defined & names, f"{f} defines {sorted(defined & names)}: import them from _capi"


def test_record_planes_match_the_kernels():
    from cygym_b200 import marl
    core = _c_constants(CORE)
    assert marl.REC_PLANES == core["CYG_REC_PLANES"]
    for p in ("P_COMP", "P_KNOWN", "P_NYA", "P_OWNED"):
        assert getattr(marl, p) == core[p], p


def test_struct_layouts_match_the_header(tmp_path):
    """sizeof and every offsetof of the six C-ABI structs, printed by a C program compiled against the header with the
    host compiler (gcc, what nvcc compiles host code with), equal the ctypes mirrors of _capi and of the oracle."""
    from cygym_b200 import _capi as K
    from oracle import cyg_oracle as O
    mirrors = [("cyg_config", K.CygConfig), ("cyg_config", O.CygConfig), ("cyg_network", K.CygNetwork),
               ("cyg_state", K.CygState), ("cyg_actions", K.CygActions), ("cyg_step_out", K.CygStepOut),
               ("cyg_rollout_args", K.CygRolloutArgs)]
    lines, expected = [], []
    for c_name, cls in mirrors:
        lines.append(f'printf("%zu\\n", sizeof({c_name}));')
        expected.append(C.sizeof(cls))
        for f in cls._fields_:
            lines.append(f'printf("%zu\\n", offsetof({c_name}, {f[0]}));')
            expected.append(getattr(cls, f[0]).offset)
    src = tmp_path / "layout.c"
    src.write_text("#include <stddef.h>\n#include <stdio.h>\n#include \"cygym_b200.h\"\nint main(void) {\n  "
                   + "\n  ".join(lines) + "\n  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-I", os.path.dirname(HEADER), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert len(got) == len(expected) >= 76
    bad = [(ln, g, e) for ln, g, e in zip(lines, got, expected) if g != e]
    assert not bad, bad


def test_config_struct_mirrors_agree():
    from cygym_b200 import _capi as K
    from oracle import cyg_oracle as O
    assert [f[0] for f in K.CygConfig._fields_] == [f[0] for f in O.CygConfig._fields_]
    assert C.sizeof(K.CygConfig) == C.sizeof(O.CygConfig)
