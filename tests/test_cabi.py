"""CPU: the C-ABI library loads and exports every symbol include/phoenix_b200.h declares (no compute calls)."""
import ctypes
import os
import re

from phoenix_b200 import _lib

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(REPO, "include", "phoenix_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(phx_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_the_expected_entry_points():
    syms = declared_symbols()
    for must in ("phx_pack_weights", "phx_rhs_forward", "phx_rhs_vjp", "phx_solve_forward", "phx_solve_adjoint",
                 "phx_stream_solve_forward", "phx_stream_solve_adjoint", "phx_ctx_create"):
        assert must in syms
    assert sorted(_lib.EXPORTS) == syms


def test_library_loads_and_exports_every_declared_symbol():
    lib = _lib.load()
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared_symbols():
        assert hasattr(raw, name), name
    assert lib.phx_resident_max_rows(0) >= 1 and lib.phx_resident_max_rows(1) >= 1
    # pure host helpers: sizes follow the documented layout
    G, H = 350, 40
    base = (2 * G * 80 + 80 + 2 * 352 + 31) // 32 * 32          # W1, WA, bias, relu(m), mask; 128-byte rounded
    Hn, KB1, GT = 48, (G + 15) // 16, (G + 127) // 128               # tensor-core operand images (phx_tc.cuh)
    images = 2 * (KB1 * 4 * Hn * 16 + GT * (2 * Hn // 16) * 2 * 128 * 16)   # forward pair + cotangent pair
    assert lib.phx_packed_bytes(G, H) == 4 * (base + images)
    assert lib.phx_tc_min_rows() == 5
    assert lib.phx_rhs_workspace_bytes(G, H, 256) > lib.phx_rhs_workspace_bytes(G, H, 4) * 2
    assert lib.phx_rhs_workspace_bytes(G, H, 7) >= 4 * (2 * 7 * 80 + 7 * G)


def test_library_exports_nothing_the_header_does_not_declare():
    """Every extern "C" phx_* symbol of the product library is part of the documented boundary (diagnostics included)."""
    import shutil
    import subprocess
    if not shutil.which("nm"):
        return
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = sorted(line.split()[-1] for line in out.splitlines()
                      if " T " in line and line.split()[-1].startswith("phx_"))
    assert exported == declared_symbols()


def test_rows_plans_for_the_baseline_shapes():
    """Host-only planning of the rows kernels: all BASELINE training shapes take 4 samples per pass; the genome-scale
    model parks its WA slice in tensor memory; the 20 000-gene sweep shape does not fit on chip (streaming engine)."""
    lib = _lib.load()
    out = (ctypes.c_int32 * 10)()
    for G, H, wa in ((350, 40, 1), (690, 40, 1), (3551, 120, 1), (11165, 40, 1), (11165, 200, 2)):
        for adj in (0, 1):
            assert lib.phx_rows_plan_describe(148, G, H, adj, out) == 0, (G, H, adj, _lib.last_error())
            assert out[6] == 4 and out[5] == wa and out[9] <= 227 * 1024 and out[8] <= 512
    assert lib.phx_rows_plan_describe(148, 20000, 200, 1, out) != 0


def test_status_struct_matches_header():
    assert ctypes.sizeof(_lib.PhxStatus) == 40


def test_solve_desc_matches_header(tmp_path):
    """The ctypes PhxSolveDesc has the size and field offsets of phx_solve_desc as a C compiler lays it out."""
    import shutil
    import subprocess
    cc = shutil.which("cc")
    if not cc:
        return
    fields = [f[0] for f in _lib.PhxSolveDesc._fields_]
    src = tmp_path / "layout.c"
    src.write_text("#include <stdio.h>\n#include <stddef.h>\n#include \"phoenix_b200.h\"\nint main(void) {\n"
                   "    printf(\"%zu\\n\", sizeof(phx_solve_desc));\n"
                   + "".join("    printf(\"%%zu\\n\", offsetof(phx_solve_desc, %s));\n" % f for f in fields)
                   + "    return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run([cc, "-I", os.path.join(REPO, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [ctypes.sizeof(_lib.PhxSolveDesc)] + [getattr(_lib.PhxSolveDesc, f).offset for f in fields]
