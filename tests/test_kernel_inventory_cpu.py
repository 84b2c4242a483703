"""CPU-side inventory of the device code in the built library (cuobjdump, no GPU): every kernel the SASS evidence script
(scripts/sass_evidence.py -> profiles/sass_*.txt) selects still exists under that template signature, the kernels
DESIGN.md calls TMA-fed really contain bulk-copy (UBLKCP) and mbarrier (SYNCS) instructions, the FP64-tensor SYRK contains
DMMA, and the whole library is built for sm_100a only.  Skipped when cuobjdump is not on PATH."""
import importlib.util
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "mir_optim_b200", "libmir_optim_b200.so")
CUOBJDUMP = shutil.which("cuobjdump") or ("/usr/local/cuda/bin/cuobjdump" if os.path.exists("/usr/local/cuda/bin/cuobjdump") else None)

pytestmark = pytest.mark.skipif(CUOBJDUMP is None or not os.path.exists(SO), reason="needs cuobjdump and the built library")


def kernel_names():
    out = subprocess.run([CUOBJDUMP, "-res-usage", SO], capture_output=True, text=True, check=True).stdout
    mangled = re.findall(r"Function (\S+):", out)
    dem = subprocess.run(["c++filt"] + mangled, capture_output=True, text=True, check=True).stdout.splitlines()
    return dict(zip(mangled, dem)), out


def opcode_counts(mangled):
    sass = subprocess.run([CUOBJDUMP, "-sass", "-fun", mangled, SO], capture_output=True, text=True).stdout
    ops = re.findall(r"/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", sass)
    return {o: ops.count(o) for o in set(ops)}


def test_library_is_sm_100a_only():
    out = subprocess.run([CUOBJDUMP, "-lelf", SO], capture_output=True, text=True, check=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_sass_evidence_selectors_match_kernels_of_the_built_library():
    spec = importlib.util.spec_from_file_location("sass_evidence", os.path.join(ROOT, "scripts", "sass_evidence.py"))
    mod = importlib.util.module_from_spec(spec); spec.loader.exec_module(mod)
    names, _ = kernel_names()
    for fname, keys in mod.KERNELS.items():
        hits = [d for d in names.values() if any(k in d for k in keys)]
        assert hits, f"{fname}: no kernel of the library matches {keys}"
        assert os.path.exists(os.path.join(ROOT, "profiles", fname)), f"profiles/{fname} is not committed"


def test_kernel_families_of_design_md_are_present():
    names, _ = kernel_names()
    dem = list(names.values())
    for family in ("lm_tpp_kernel", "lm_small_kernel", "lm_mux_kernel", "lm_cta_kernel", "boxqp_cta_kernel", "boxqp_warp_kernel",
                   "syrk_dmma_kernel", "large_jac_kernel", "large_ctl_mid_kernel", "large_ctl_post_kernel"):
        assert any(family in d for d in dem), family


def test_tma_fed_kernels_contain_bulk_copies_and_mbarriers():
    names, _ = kernel_names()
    by_dem = {d: m for m, d in names.items()}
    syrk = next(m for d, m in by_dem.items() if "syrk_dmma_kernel" in d)
    ops = opcode_counts(syrk)
    assert ops.get("DMMA", 0) > 100 and ops.get("UBLKCP", 0) > 0 and ops.get("SYNCS", 0) > 0, ops
    spline = next(m for d, m in by_dem.items() if "lm_cta_kernel<mirb200::CtaSpline<double>, double, true>" in d)
    ops = opcode_counts(spline)
    assert ops.get("UBLKCP", 0) > 0 and ops.get("SYNCS", 0) > 0, ops


def test_headline_kernel_loads_slab_into_registers_and_evaluates_both_exp_pairs():
    # DESIGN.md section 7: the row loop of the thread-per-problem kernel keeps its slab prefetch in registers (no cp.async,
    # LDGSTS) and evaluates the exps of a row pair at the trial point and at the anchor
    names, _ = kernel_names()
    tpp = next(m for m, d in names.items() if "lm_tpp_kernel<mirb200::ModelGauss4<double, true>, double, false, true, true>" in d)
    ops = opcode_counts(tpp)
    assert ops.get("LDGSTS", 0) == 0, ops
    assert ops.get("DFMA", 0) > 300, ops          # two interleaved exp pairs per row pair
