"""The C-ABI library loads without a GPU and exports every symbol include/*.h declares."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "graphpope_b200.h")


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"^\s*(?:const\s+)?(?:int64_t|int|char)\s*\*?\s*(gp_[a-z0-9_]+)\s*\(", src, flags=re.M)
    return sorted(set(names))


def test_header_declares_the_expected_surface():
    names = declared_functions()
    for must in ("gp_csr_build", "gp_msbfs_run", "gp_msbfs_features", "gp_normalize_into",
                 "gp_geodesic_embed_host", "gp_degree", "gp_pagerank", "gp_topk_stable_f64",
                 "gp_cdist_minmax", "gp_decode_gathered", "gp_last_error"):
        assert must in names
    assert len(names) >= 36


def test_library_exports_every_declared_symbol():
    from graphpope_b200 import _lib

    assert os.path.exists(_lib.LIB_PATH), "build the library first: __graft_entry__.build()"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared_functions():
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert set(declared_functions()) == set(_lib.SIGNATURES), "ctypes table out of sync with the header"


def test_no_compute_without_gpu_but_clean_errors():
    import torch

    from graphpope_b200 import _lib

    lib = _lib.load()
    assert lib.gp_abi_version() == 1
    assert lib.gp_status_string(5) == b"hop distance does not fit uint16"
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            _lib.require_cuda()
        assert lib.gp_device_info(None, None, None, None, 0) == _lib.GP_ERR_NO_DEVICE
        assert b"no CUDA device" in lib.gp_last_error()
    # argument checks come before any CUDA call
    assert lib.gp_betweenness(None, None, None) == _lib.GP_ERR_INVALID
    assert lib.gp_eigenvector(None, 1e-15, 10, None, None, None) == _lib.GP_ERR_INVALID
    assert lib.gp_concat_x(None, 4, 4, 2, None, 8, None) == _lib.GP_ERR_INVALID  # ld_x < F
    assert lib.gp_concat_x(None, 0, 4, 4, None, 8, None) == _lib.GP_OK            # nothing to copy
    # round 1's pull exchange: exported for ABI 1 callers, refused without touching the device
    removed = {
        "gp_msbfs_pack": (None, 0, None, None, None, None, None, None),
        "gp_geodesic_run_packed": (None, None, None, 0, None, 0, 0, None),
        "gp_msbfs_packed_info": (None, 0, None, None, None, None, None),
        "gp_msbfs_ipc_export": (None, None, None),
        "gp_decode_peers": (None, 0, 0, 0, 0, 0, 0, None, 0, 0, None, 0, 0, None),
    }
    for name, args in removed.items():
        assert getattr(lib, name)(*args) == _lib.GP_ERR_UNSUPPORTED, name
        assert lib.gp_last_error() == f"{name}: removed, use gp_geodesic_run_exchange".encode(), name


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "graphpope_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "/root/reference" not in text, f


def test_plain_c_caller_compiles_and_runs(tmp_path):
    """examples/embed_host.c: the boundary from strict C99, no Python / torch in the process.  With a B200 it checks
    its own rows (exit 0); without one the library must answer GP_ERR_NO_DEVICE cleanly (exit 2), not crash."""
    import shutil
    import subprocess

    from graphpope_b200 import _lib

    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    libdir = os.path.dirname(_lib.LIB_PATH)
    exe = str(tmp_path / "embed_host")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "examples", "embed_host.c"), "-L", libdir, "-lgraphpope_b200",
                    f"-Wl,-rpath,{libdir}", "-o", exe], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert "graphpope_b200 ABI 1" in r.stdout
    if r.returncode == 0:
        assert "6 nodes x (2 features + 4 anchors): ok" in r.stdout
    else:
        assert r.returncode == 2 and "no CUDA device" in r.stdout, r.stdout + r.stderr


def test_sass_is_sm_100a_with_the_blackwell_paths_it_claims():
    """The in-tree library holds sm_100a code only, and the instructions DESIGN.md names are really in it:
    tcgen05.mma / commit / ld (cdist), the bulk-copy engine + mbarriers (exchange, x copy), 256-bit loads (MS-BFS)."""
    import shutil
    import subprocess

    from graphpope_b200 import _lib

    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("no cuobjdump")
    elfs = subprocess.run([cuobjdump, "-lelf", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    archs = set(re.findall(r"\.(sm_\w+)\.cubin", elfs))
    assert archs == {"sm_100a"}, archs
    sass = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    per_kernel, cur = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            per_kernel[cur] = set()
            continue
        for mnem in ("UTCHMMA", "UTCBAR", "LDTM", "UBLKCP", "SYNCS", "LDG.E.ENL2.256", "HMMA.", "WGMMA"):
            if cur is not None and mnem in line:
                per_kernel[cur].add(mnem)

    def used_by(fragment):
        got = set()
        for name, mn in per_kernel.items():
            if fragment in name:
                got |= mn
        return got

    assert {"UTCHMMA", "UTCBAR", "LDTM", "SYNCS"} <= used_by("cdist_kernel")
    assert {"UBLKCP", "SYNCS"} <= used_by("exchange_decode_kernel")
    assert {"UBLKCP", "SYNCS"} <= used_by("xcopy_tma_kernel")
    assert "LDG.E.ENL2.256" in used_by("msbfs_kernel")
    assert not any("WGMMA" in mn for mn in per_kernel.values())  # sm_90a-only; must not appear
