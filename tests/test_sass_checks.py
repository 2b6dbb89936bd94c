"""Static checks on the SASS of the built library (no GPU needed): the step kernel really uses tensor memory, and the
bank-conflict counter (tools/sass_bank_conflicts.py) finds the four solver loops."""
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def sass(tmp_path_factory):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    import __graft_entry__ as ge
    ge.build()
    out = tmp_path_factory.mktemp("sass") / "lib.sass"
    with open(out, "w") as f:
        subprocess.check_call([exe, "-sass", os.path.join(ROOT, "bullet_envs_b200", "csrc", "libsnake_b200.so")], stdout=f)
    return str(out)


def test_hybrid_step_kernel_uses_tensor_memory_shared_memory_and_registers(sass):
    """the benchmarked kernel (RowsH): 8 / 4 / 2 word tensor-memory loads, tensor-memory stores of the solver state, the three
    shared-memory loads of the friction record, and a fully unrolled normal sweep (one 4-word load per contact)"""
    txt = open(sass).read()
    k = [p for p in txt.split("Function : ") if p.startswith("_Z19snk_hyb_step_kernelILb1ELb0ELb0EE")][0]
    assert k.count("LDTM.x8") >= 3 and k.count("LDTM.x4") >= 32 and k.count("LDTM.x2") >= 32
    assert k.count("STTM.x2") >= 3 and k.count("STTM.x8") >= 2
    assert k.count("LDS.128") >= 3 and k.count("LDS.64") >= 3


def test_bank_conflict_counter_finds_the_solver_loops(sass):
    """tools/sass_bank_conflicts.py on the hybrid kernel: the rolled friction loop (2 pairs per iteration, MUFU of the cone projection,
    tensor-memory loads) is found, and its register-bank conflicts per pair stay below the first version's 17.7 per contact and sweep"""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import sass_bank_conflicts as sbc
    k = sbc.kernels(sass)
    name = [n for n in k if "snk_hyb_step_kernelILb1ELb0ELb0EE" in n][0]
    found = []
    for body in sbc.loops(sbc.ins_of(k[name])):
        if 100 <= len(body) <= 200 and any("LDTM.x8" in t for _, t in body) and sum("MUFU.RSQ" in t for _, t in body) == 2:
            found.append((len(body),) + sbc.metric(body))
    assert len(found) == 1, found
    n, conflicts, reuse, nfp = found[0]
    assert n <= 150 and conflicts / 2 < 17.7, found


def test_manifold_kernel_streams_rows_with_async_copies(sass):
    """snk_man_step_kernel: the solver sweeps fill their shared-memory ring with cp.async (LDGSTS, 16 bytes, L2 only) and wait per group
    (LDGDEPBAR / DEPBAR); no tensor-memory instruction (the kernel has no warp-convergence requirement)"""
    txt = open(sass).read()
    k = [p for p in txt.split("Function : ") if p.startswith("_Z19snk_man_step_kernelILb1EE")][0]
    assert k.count("LDGSTS") >= 12, k.count("LDGSTS")          # 2 words per normal row + 4 per friction row, prologue + loop
    assert "LDGDEPBAR" in k and "DEPBAR" in k
    assert "LDTM" not in k and "STTM" not in k


def test_bullet_order_kernel_is_a_branch_free_block_sweep(sass):
    """snk_env_kernel (motor_solver = 0): the block Gauss-Seidel broadcasts one impulse change per row with an indexed shuffle (no
    butterfly in the solver loops: SHFL.BFLY would be the round-1 reduction) and selects instead of branching on the clamps"""
    txt = open(sass).read()
    k = [p for p in txt.split("Function : ") if p.startswith("_Z14snk_env_kernelI10WarpMemPgsLb0ELi1ELi9EE")][0]
    assert k.count("SHFL.IDX") >= 20 and k.count("SHFL.BFLY") <= 8, (k.count("SHFL.IDX"), k.count("SHFL.BFLY"))
    assert k.count("REDUX") >= 1                                # the residual's warp maximum
