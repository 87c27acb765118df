"""T6 build hygiene (SURVEY section 4), no GPU needed: the built library is sm_100a code with the instruction forms the
design relies on -- 128-bit global accesses in the step kernel, packed FFMA2 in the fp32 rollout, FP64 FMAs in the fp64
one, programmatic-dependent-launch instructions, no register spills in the rollout kernels."""
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import sass_stats  # noqa: E402

from abi_support import ptxas_blocks  # noqa: E402
from random_envs_b200 import build as lib_build  # noqa: E402


@pytest.fixture(scope="module")
def sass():
    lib_build.build()
    return sass_stats.functions(lib_build.LIB_PATH)


def _ops(rows):
    return [op for _, op, _ in rows]


def _one(sass, *needles):
    hits = [name for name in sass if all(n in name for n in needles)]
    assert len(hits) == 1, (needles, hits)
    return sass[hits[0]]


def test_library_targets_sm_100a_only():
    out = subprocess.run(["cuobjdump", "-lelf", lib_build.LIB_PATH], stdout=subprocess.PIPE, text=True, check=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_step_kernel_uses_128_bit_accesses_and_programmatic_dependent_launch(sass):
    ops = _ops(_one(sass, "cartpole_step_kernelIfLb1ELb0ELb0"))    # <float, auto_reset, not noisy, not lean>
    assert sum(o.startswith("LDG.E.128") for o in ops) >= 9        # 4 state rows + 4 xi rows + elapsed
    assert sum(o.startswith("STG.E.128") for o in ops) >= 6        # 4 state rows + elapsed + reward
    assert "ACQBULK" in ops and "PREEXIT" in ops                   # griddepcontrol.wait / launch_dependents
    # tile-granular step ordering: ticket atomic, acquire poll, release store, L2 bulk prefetch of the tile
    assert any(o.startswith("ATOMG.E.ADD.STRONG.GPU") for o in ops) and any(o.startswith("LDG.E.STRONG.GPU") for o in ops)
    assert any(o.startswith("STG.E.STRONG.GPU") for o in ops) and sum(o.startswith("UBLKPF") for o in ops) >= 4
    lean = _ops(_one(sass, "cartpole_step_kernelIfLb1ELb0ELb1"))   # lean step: 64-bit load / store of four uint16 counters
    assert any(o.startswith("LDG.E.64") for o in lean) and any(o.startswith("STG.E.64") for o in lean)
    ops64 = _ops(_one(sass, "cartpole_step_kernelIdLb1ELb0ELb0"))
    assert sum(o.startswith("LDG.E.128") for o in ops64) >= 10 and any(o.startswith("DFMA") for o in ops64)


def test_fp32_rollout_runs_on_the_packed_fp32_pipe_and_fp64_rollout_on_dfma(sass):
    pair = _ops(_one(sass, "cartpole_rollout_pair_kernelILb1"))
    assert sum(o.startswith("FFMA2") for o in pair) >= 100 and sum(o.startswith("FMUL2") for o in pair) >= 50
    f64 = _ops(_one(sass, "cartpole_rollout_kernelIdLb1ELb0ELb0"))
    assert sum(o.startswith("DFMA") for o in f64) > 500 and not any(o.startswith("FFMA2") for o in f64)


def test_uniform_sampler_loop_is_philox_plus_conversion_only(sass):
    rows = _one(sass, "dr_sample_f32_kernelILi1ELi0")               # <uniform, 128-bit stores>
    ops = _ops(rows)
    assert 17 <= sum(o.startswith("IMAD.WIDE.U32") for o in ops) <= 24    # Philox4x32-10 with the first rounds' constants hoisted
    assert not any(o.startswith("F2F") for o in ops)               # parameters arrive converted (host side)
    assert sum(o.startswith("FFMA2") for o in ops) >= 2            # packed affine map
    assert any(o.startswith("STG.E.128") for o in ops)
    assert not any(o.startswith(("STL", "LDL")) for o in ops)      # no stack traffic
    for kind in ("Li2ELi1", "Li3ELi1"):                            # truncnorm / gaussian, 30-dim store shape
        tn = _ops(_one(sass, "dr_sample_f32_kernelI" + kind))
        assert sum(o.startswith("FFMA2") for o in tn) >= 2 and sum(o.startswith("FMUL2") for o in tn) >= 2
    f64 = _ops(_one(sass, "dr_sample_kernelIdLi1ELi0"))             # fp64 keeps the generic kernel
    assert sum(o.startswith("IMAD.WIDE.U32") for o in f64) >= 19


def test_fullgaussian_contraction_runs_on_tcgen05(sass):
    """The one GEMM-shaped op of the path: UTC*MMA (tcgen05.mma), STTM / LDTM (tcgen05.st / .ld), TMEM allocation."""
    ops = _ops(_one(sass, "dr_sample_fullgaussian_tc_kernel"))
    assert sum(o.startswith("UTCHMMA") for o in ops) == 12         # 4 K-steps x 3 (head/tail split) per 128-sample tile
    assert sum(o.startswith("STTM") for o in ops) >= 8 and sum(o.startswith("LDTM") for o in ops) >= 1
    assert any(o.startswith("UTCBAR") for o in ops)                # tcgen05.commit -> mbarrier
    assert not any(o.startswith(("HMMA", "STL", "LDL")) for o in ops)


def test_no_register_spills_in_any_kernel():
    """Every kernel of the library: zero spill stores / loads (ptxas -v log written by the build)."""
    blocks = ptxas_blocks()
    assert len(blocks) >= 45
    seen = set()
    for name, b in blocks.items():
        for st, ld in re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", b):
            assert st == "0" and ld == "0", (name, st, ld)
        regs = int(re.search(r"Used (\d+) registers", b).group(1))
        if "rollout_pair" in name or ("rollout_kernelId" in name and name.endswith("ELb0ELb0EEEvNS_11RolloutArgsIT_EE")):
            assert regs <= 80, (name, regs)                          # 3 CTAs of 256 threads per SM
        if "cartpole_step_kernelIfLb1ELb0" in name:
            assert regs <= 64, (name, regs)                          # 4 CTAs of 256 threads per SM
        seen.add(name.split("IL")[0][:40])
    assert len(seen) >= 8
