"""The C-ABI boundary without a GPU: libsimstep.so builds, loads and exports exactly what include/simstep.h
declares; the ctypes structs mirror the header; and the product path fails loudly (no CPU fallback)."""
import ctypes as C
import os
import re

import pytest
import torch

from amp_extensions_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "simstep.h")


def header_text():
    with open(HEADER) as f:
        return f.read()


def declared_functions():
    return sorted(set(re.findall(r"\b(simstep_[a-z0-9_]+)\s*\(", header_text())))


def test_library_builds_in_tree_for_sm_100a():
    lib = build.build()
    assert os.path.exists(lib) and os.path.dirname(lib).endswith(os.path.join("amp_extensions_b200", "csrc"))
    assert "arch=compute_100a,code=sm_100a" in " ".join(build.NVCC_FLAGS) and "-lineinfo" in build.NVCC_FLAGS


def test_every_declared_symbol_is_exported_and_bound():
    names = declared_functions()
    assert len(names) >= 20
    raw = C.CDLL(_lib.lib_path())
    for n in names:
        assert hasattr(raw, n), f"{n} is declared in simstep.h but not exported by libsimstep.so"
    assert sorted(_lib.EXPORTED_SYMBOLS) == names, "ctypes binding and header disagree"


def test_abi_version_and_constants_match_header():
    h = header_text()
    lib = _lib.load(build_if_missing=False)
    assert lib.simstep_abi_version() == int(re.search(r"#define SIMSTEP_ABI_VERSION (\d+)", h).group(1)) == _lib.ABI_VERSION
    for macro, val in (("SIMSTEP_MAX_HIDDEN", _lib.MAX_HIDDEN), ("SIMSTEP_MAX_BODIES", _lib.MAX_BODIES),
                       ("SIMSTEP_MAX_JOINTS", _lib.MAX_JOINTS)):
        assert int(re.search(rf"#define {macro} (\d+)", h).group(1)) == val
    for name, code in _lib.PREC.items():
        assert int(re.search(rf"#define SIMSTEP_PREC_{name.upper()} (\d+)", h).group(1)) == code
    for name, code in _lib.RFF_INPUT.items():
        assert int(re.search(rf"#define SIMSTEP_RFF_INPUT_{(name or 'auto').upper()} (\d+)", h).group(1)) == code
    n_cat = int(re.search(r"#define SIMSTEP_PROF_CATEGORIES (\d+)", h).group(1))
    assert len(_lib.PROF_CATEGORIES) == n_cat


def test_struct_sizes_match_the_c_layout():
    # all members are 4-byte scalars or arrays of them: size = 4 * number of scalar slots, no padding
    assert C.sizeof(_lib.SimstepConfig) == 4 * (5 + _lib.MAX_HIDDEN + 5 + 7)
    assert C.sizeof(_lib.SimstepTermination) == 4 * (8 + 4 * _lib.MAX_BODIES + 1)
    # n_joints, dof + six per-joint scalars + two per-joint 3-vectors
    assert C.sizeof(_lib.SimstepCharacter) == 4 * (2 + 6 * _lib.MAX_JOINTS + 2 * 3 * _lib.MAX_JOINTS)


def test_no_torch_types_cross_the_boundary():
    h = header_text()
    assert "torch" not in h.replace("no torch", "") and "at::" not in h and "std::" not in h
    assert 'extern "C"' in h


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_product_path_fails_loudly_without_a_gpu():
    """There is no CPU fallback: creating a handle, an Engine or stepping an env without a device raises."""
    lib = _lib.load(build_if_missing=False)
    cfg = _lib.SimstepConfig()
    cfg.abi_version, cfg.state_dim, cfg.action_dim, cfg.n_models, cfg.n_hidden = _lib.ABI_VERSION, 8, 2, 2, 1
    cfg.hidden[0] = 16
    h = C.c_void_p()
    rc = lib.simstep_create(C.byref(cfg), C.byref(h))
    assert rc in (-3, -2) and not h.value
    assert lib.simstep_last_error(None)
    from amp_extensions_b200 import Engine
    with pytest.raises(_lib.SimstepError):
        Engine(8, 2, 2, [16])


def test_create_rejects_bad_arguments_before_touching_the_device():
    lib = _lib.load(build_if_missing=False)
    h = C.c_void_p()
    cfg = _lib.SimstepConfig()
    cfg.abi_version = _lib.ABI_VERSION + 1
    assert lib.simstep_create(C.byref(cfg), C.byref(h)) == -1
    assert b"abi_version" in lib.simstep_last_error(None)
    cfg.abi_version = _lib.ABI_VERSION
    cfg.state_dim, cfg.n_models = 0, 4
    assert lib.simstep_create(C.byref(cfg), C.byref(h)) == -1
    cfg.state_dim, cfg.n_models = 8, 9
    assert lib.simstep_create(C.byref(cfg), C.byref(h)) == -1
    assert lib.simstep_create(None, C.byref(h)) == -1
    # NULL handles never crash
    assert lib.simstep_destroy(None) == 0
    assert lib.simstep_step(None, None, None, None, None, 0, None, None, None, None) == -1


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "amp_extensions_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".inc", ".h")):
                with open(os.path.join(dirpath, f)) as fh:
                    src = fh.read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f"{f} imports the oracle"


def test_native_code_reads_only_the_documented_environment_switches():
    """The library reads three environment variables (README.md, "Diagnostic switches"): SIMSTEP_CHAIN=0 forces one
    launch per layer, SIMSTEP_IMIT_GENERIC=1 the generic imitation kernel, SIMSTEP_DEBUG_GUARDS=1 the workspace guard
    zones.  A selection between kernels is made from the inputs, not left to a variable set by the user."""
    csrc = os.path.join(ROOT, "amp_extensions_b200", "csrc")
    calls, names = 0, []
    for f in sorted(os.listdir(csrc)):
        if f.endswith((".cu", ".cuh", ".inc", ".h")):
            with open(os.path.join(csrc, f)) as fh:
                src = fh.read()
            calls += src.count("getenv(")
            names += re.findall(r'getenv\(\s*"([A-Za-z0-9_]+)"\s*\)', src)
    assert calls == len(names), "every getenv call names its variable literally"
    assert set(names) == {"SIMSTEP_CHAIN", "SIMSTEP_IMIT_GENERIC", "SIMSTEP_DEBUG_GUARDS"}, sorted(names)


def test_forward_kernel_schedule_covers_every_unit_exactly_once():
    """The column-fused forward kernel's unit schedule (csrc/gemm_chain.cuh: chain_schedule + chain_item, evaluated on
    the HOST through simstep_debug_chain_schedule - no GPU involved): for every batch / ensemble shape each
    (env tile, member) unit is run exactly once as a whole or exactly once by each of the two roles of a shared unit;
    shared units only exist in the last round, on pairs 2u and 2u + 1, and number at most half the pairs; whole rounds
    of members-in-sequence keep an env tile's members on one pair, in order; no pair gets more than one item more than
    its share."""
    lib = _lib.load(build_if_missing=False)
    max_items = 4096
    buf = (C.c_int32 * (74 * max_items * 2))()
    pairs, seq, tail = C.c_int32(), C.c_int32(), C.c_int32()
    shapes = [(m, g, sm) for g in (1, 2, 3, 4, 5, 8) for m in (1, 2, 9, 18, 19, 37, 73, 74, 75, 83, 148, 157, 256, 300)
              for sm in (148,)] + [(157, 4, 132), (40, 4, 8), (5, 3, 2), (1000, 1, 148), (511, 7, 148)]
    for m_tiles, groups, sm in shapes:
        rc = lib.simstep_debug_chain_schedule(m_tiles, groups, sm, max_items, C.byref(pairs), C.byref(seq), C.byref(tail), buf)
        assert rc == 0, (m_tiles, groups, sm)
        P, R, T = pairs.value, seq.value, tail.value
        units = m_tiles * groups
        assert P == min(units, sm // 2) and 0 <= 2 * T <= P and R == (m_tiles // P if units > P else 0)
        whole, roles, counts = {}, {}, []
        for p in range(P):
            items = []
            for i in range(max_items):
                u, r = buf[(p * max_items + i) * 2], buf[(p * max_items + i) * 2 + 1]
                if u < 0:
                    break
                items.append((u, r))
            counts.append(len(items))
            for i, (u, r) in enumerate(items):
                assert 0 <= u < units
                if r < 0:
                    assert u not in whole and u not in roles, (m_tiles, groups, u)
                    whole[u] = (p, i)
                else:
                    assert i == len(items) - 1 and p < 2 * T and r == p % 2 and u == units - T + p // 2
                    assert (u, r) not in roles and u not in whole
                    roles[(u, r)] = p
            # rounds of members in sequence: the first R * groups items walk R env tiles member by member
            for k in range(R):
                tile = p + k * P
                assert items[k * groups:(k + 1) * groups] == [(tile * groups + g, -1) for g in range(groups)]
        assert len(whole) == units - T and len(roles) == 2 * T, (m_tiles, groups, sm, len(whole), len(roles))
        assert all((units - T + j, r) in roles for j in range(T) for r in (0, 1))
        assert max(counts) - min(counts) <= 1 or T > 0 and max(counts) - min(counts) <= 2
