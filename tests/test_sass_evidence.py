"""What the compiled library contains, checked on the CPU from its SASS (cuobjdump): the design claims of DESIGN.md that can
be read off the machine code -- the Gram kernel runs on the FP64 tensor pipe (DMMA.8x8x4) fed by the TMA engine (UBLKCP)
through mbarriers (SYNCS), the data-flow Cholesky factorisation runs its tile updates on DMMA too and factorises its diagonal
blocks in registers with shuffles, the E-step sweeps are pure DFMA with the table look-up in shared memory and no
local-memory spill, and every kernel is built for sm_100a.  No GPU."""
import collections
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "gingr_b200", "lib", "libgingr_cuda.so")
pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="no cuobjdump")


@pytest.fixture(scope="module")
def kernels():
    if not os.path.exists(LIB):
        from gingr_b200 import build
        build.build()
    out = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    archs = set(re.findall(r"arch = (sm_\w+)", out))
    table = {}
    for block in re.split(r"\n\s*Function : ", out)[1:]:
        name = block.split("\n", 1)[0].strip()
        c = collections.Counter(re.findall(r"^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_]*(?:\.[A-Z0-9_x]+)*)", block, flags=re.M))
        table[name] = c
    return archs, table


def _find(table, fragment):
    hits = [k for k in table if fragment in k]
    assert hits, fragment
    return hits


def _count(counter, prefix):
    return sum(v for k, v in counter.items() if k == prefix or k.startswith(prefix + "."))


def test_everything_is_built_for_sm_100a(kernels):
    archs, table = kernels
    assert archs == {"sm_100a"}, archs
    assert len(table) >= 80


def test_gram_kernel_is_dmma_fed_by_tma_through_mbarriers(kernels):
    _, table = kernels
    for name in _find(table, "gram_ws_kernel"):
        c = table[name]
        assert _count(c, "DMMA") >= 256 and any(k.startswith("DMMA.8x8x4") for k in c)
        assert _count(c, "UBLKCP") >= 1                      # cp.async.bulk: the TMA engine moves the operand rows
        assert _count(c, "SYNCS") >= 4                       # mbarrier arrive / try_wait on the full and empty rings
        assert _count(c, "DFMA") == 0 and _count(c, "LDL") == 0 and _count(c, "STL") == 0


def test_estep_sweeps_are_spill_free_dfma_with_the_table_in_shared_memory(kernels):
    _, table = kernels
    for frag in ("estep_colsum_kernel", "estep_rowsum_kernel"):
        for name in _find(table, frag):
            c = table[name]
            assert _count(c, "DFMA") >= 300 and _count(c, "LDS") >= 30
            assert _count(c, "LDL") == 0 and _count(c, "STL") == 0          # no local-memory traffic in the hot loops
            assert _count(c, "DMMA") == 0


def test_cholesky_tiles_are_dmma_and_diagonal_blocks_factorise_in_registers_with_shuffles(kernels):
    _, table = kernels
    names = _find(table, "chol_df_kernel")
    assert len(names) == 2, names                               # the single and the batched form
    for name in names:
        c = table[name]
        assert _count(c, "DMMA") >= 64 and _count(c, "SHFL") >= 32
        assert _count(c, "LDL") == 0 and _count(c, "STL") == 0


def test_every_kernel_of_the_mh_step_has_a_batched_twin(kernels):
    """csrc/batch.cuh: the kernels on the path of a Metropolis-Hastings step / an ICP iteration exist twice in the library --
    `name` (arguments in the parameter bank) and `name_batched` (blockIdx.z = chain, arguments from an array) -- generated
    from one body, so the twin carries the same arithmetic (the compiler may unroll the two differently: the check is on the
    kind of arithmetic -- FP64 pipe, FP64 tensor instructions -- not on instruction counts)."""
    _, table = kernels
    names = ["multi_copy_kernel", "add_normal_kernel", "chol_backsolve_small_kernel", "chol_small_kernel", "dense_matvec_kernel",
             "combine_kernel", "gemv_rows_kernel", "procrustes_sums_kernel", "procrustes_reduce_then_kernel", "coeff_residual_kernel",
             "gemvT_kernel", "gemvT_reduce_kernel", "finalize_kernel", "mcmc_random_override_kernel", "fit_from_instance_kernel",
             "pose_kernel", "vertex_normals_kernel", "surface_kernel", "surface_reduce_kernel", "mean_sqrt_kernel", "nn_vertex_kernel",
             "nn_reduce_kernel", "line_mesh_kernel", "icp_weights_kernel", "obs_kernel", "sigma2_kernel", "gram_ws_kernel",
             "gram_finish_kernel", "chol_df_kernel", "mcmc_residual_kernel", "mcmc_build_system_kernel", "mcmc_quadform_kernel",
             "mcmc_distance_logpdf_kernel", "mcmc_decide_kernel", "mcmc_restore_ints_kernel", "bump_iteration_kernel"]

    def fp(counter):
        return (_count(counter, "DFMA") + _count(counter, "DMUL") + _count(counter, "DADD"), _count(counter, "DMMA"))
    for n in names:
        single = [k for k in table if re.search(r"\d+" + n + r"(E|I)", k) and "_batched" not in k]
        twin = [k for k in table if re.search(r"\d+" + n + r"_batched(E|I)", k)]
        assert single and twin, n
        assert len(single) == len(twin), (n, single, twin)          # template kernels: one twin per instantiation
        kinds = lambda ks: sorted((a > 0, b > 0) for a, b in (fp(table[k]) for k in ks))
        assert kinds(single) == kinds(twin), n


def test_small_matrix_factorisation_fits_two_ctas_per_sm():
    """chol_small_kernel (one 64 x 64 block; what 1024 batched chains of rank 50 factorise twice per MH step): at most 128
    registers and no local memory in both forms, so that two CTAs of 256 threads share an SM -- the data-flow kernel it
    replaces for n <= 64 needs 214 registers (one CTA per SM)."""
    out = subprocess.run(["cuobjdump", "--dump-resource-usage", LIB], capture_output=True, text=True, check=True).stdout
    usage = {}
    name = None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", line)
        if m and name:
            usage[name] = tuple(int(v) for v in m.groups())
            name = None
    small = {k: v for k, v in usage.items() if "chol_small_kernel" in k}
    assert len(small) == 2, list(small)
    for k, (reg, stack, shared, local) in small.items():
        assert reg <= 128 and stack == 0 and local == 0, (k, reg, stack, local)
    big = [v for k, v in usage.items() if "chol_df_kernel" in k and "batched" not in k]
    assert big and big[0][0] > 128
