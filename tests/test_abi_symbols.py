"""CPU-side check of the drop-in boundary: the shared library loads without a GPU and exports
every function `include/b200rdo.h` declares (parsed from the header, macro-generated per-size
symbols included); creating a context without a device fails loudly with B200_ERR_NODEV."""
import ctypes as C
import os
import re

from rav1e_b200 import backend as B

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    """Every function the header declares, macro-generated families included: the header is run
    through the C preprocessor (gcc -E) and every prototype name is collected."""
    import subprocess
    src = subprocess.run(["gcc", "-E", "-P", os.path.join(ROOT, "include", "b200rdo.h")], check=True,
                         capture_output=True, text=True).stdout
    names = set(re.findall(r"\b((?:b200|rav1e)_[A-Za-z0-9_]+)\s*\(", src))
    return sorted(names)


def reference_table_symbols():
    """The names the reference binds for this path, written out from its tables with the ISA suffix
    replaced by `_cuda`."""
    names = set()
    # asm/x86/dist/mod.rs:21-43, tables :483-729 (22 BlockSize variants, partition.rs:130-153)
    for w, h in B.BLOCK_SIZES:
        names |= {f"rav1e_sad{w}x{h}_cuda", f"rav1e_sad_{w}x{h}_hbd_cuda", f"rav1e_satd_{w}x{h}_cuda",
                  f"rav1e_satd_{w}x{h}_hbd_cuda"}
    # asm/x86/mc.rs:394-405 (put), :424-435 (put hbd), :508-519 (prep), :563-574 (prep hbd), :582-620 (avg)
    filters = ["8tap_regular", "8tap_regular_smooth", "8tap_regular_sharp", "8tap_smooth_regular", "8tap_smooth",
               "8tap_smooth_sharp", "8tap_sharp_regular", "8tap_sharp_smooth", "8tap_sharp", "bilin"]
    for f in filters:
        for kind in ("put", "prep"):
            for bpc in (8, 16):
                names.add(f"rav1e_{kind}_{f}_{bpc}bpc_cuda")
    names |= {"rav1e_avg_8bpc_cuda", "rav1e_avg_16bpc_cuda"}
    # asm/x86/predict.rs:36-120 (angular), :125-141 (z2), :157-186 (cfl_ac), :203-234 (cfl)
    modes = ["h", "v", "dc", "dc_left", "dc_128", "dc_top", "smooth_v", "smooth_h", "smooth", "z1", "z2", "z3",
             "paeth", "cfl", "cfl_left", "cfl_top", "cfl_128", "cfl_ac_420", "cfl_ac_422", "cfl_ac_444"]
    for m in modes:
        for bpc in (8, 16):
            names.add(f"rav1e_ipred_{m}_{bpc}bpc_cuda")
    # asm/x86/cdef.rs:146-167 (filter), :236-260 (dir)
    names |= {f"rav1e_cdef_filter_{s}_cuda" for s in ("4x4", "4x8", "8x8")}
    names |= {"rav1e_cdef_dir_8bpc_cuda", "rav1e_cdef_dir_16bpc_cuda"}
    return names


def test_library_exports_every_declared_symbol():
    L = C.CDLL(B.LIB_PATH)
    syms = declared_symbols()
    assert len(syms) >= 60 + 88 + 42 + 40 + 5
    missing = [s for s in syms if not hasattr(L, s)]
    assert not missing, missing
    assert L.b200_abi_version() == 1


def test_every_reference_table_entry_has_its_cuda_symbol():
    """SAD_FNS / SATD_FNS / PUT_FNS / PREP_FNS / AVG_FNS / the ipred symbols / CDEF_FILTER_FNS /
    CDEF_DIR_*_FNS: every extern the reference declares for the path is declared in the header with
    the `_cuda` suffix and exported by the library."""
    L = C.CDLL(B.LIB_PATH)
    declared = {s for s in declared_symbols() if s.startswith("rav1e_")}
    want = reference_table_symbols()
    assert want <= declared, sorted(want - declared)
    # nothing under the reference's prefix that the reference does not have, except the HBD CDEF
    # filters (the reference's HBD table is empty, asm/x86/cdef.rs:174-178)
    extra = declared - want
    assert extra == {f"rav1e_cdef_filter_{s}_16bpc_cuda" for s in ("4x4", "4x8", "8x8")}, sorted(extra)
    assert all(hasattr(L, s) for s in want)


def test_no_device_is_a_loud_error_not_a_fallback():
    """Run in a child process that sees no CUDA device (an empty CUDA_VISIBLE_DEVICES hides those of a GPU machine)."""
    import subprocess
    import sys
    code = ("from rav1e_b200 import backend as B\n"
            "try:\n    B.Context(0)\n    print('created')\n"
            "except B.B200Error as e:\n    print(e.status, e)\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), timeout=120)
    assert r.returncode == 0, r.stderr
    status, msg = r.stdout.split(" ", 1)
    assert int(status) == B.ERR_NODEV
    assert "no CPU fallback" in msg


def test_header_block_sizes_match_the_reference_list():
    """22 BlockSize variants (partition.rs:130-153) — the table the asm wrappers index."""
    assert len(B.BLOCK_SIZES) == 22 and len(set(B.BLOCK_SIZES)) == 22
    L = B.lib()
    assert [L.b200_tx_width(i) for i in range(5)] == [4, 8, 16, 32, 64]
    assert (L.b200_tx_width(17), L.b200_tx_height(17)) == (16, 64)
    assert L.b200_valid_av1_transform(4, 0) == 1 and L.b200_valid_av1_transform(4, 1) == 0
