"""CPU: the C-ABI library loads and exports every symbol the header declares; host-side logic
(theta solver, column sharding, LIBSVM parser, constructors' RNG order) without touching a GPU."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from oracle import accbpg_oracle as orc


def test_library_exports_every_declared_symbol():
    from accbpg_and_fw_b200 import _native as nat
    assert os.path.exists(nat.LIB_PATH)
    header = open(os.path.join(ROOT, "include", "accbpg_b200.h")).read()
    declared = set(re.findall(r"\b(accbpg_\w+)\s*\(", re.sub(r"/\*.*?\*/", " ", header, flags=re.S)))
    assert len(declared) >= 40
    assert declared == set(nat.PROTOS), declared ^ set(nat.PROTOS)
    raw = ctypes.CDLL(nat.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), name
    assert nat.lib.accbpg_abi_version() == nat.MACROS["ACCBPG_ABI_VERSION"]
    assert nat.launch_count() == 0            # nothing computed on CPU
    nm = subprocess.run(["nm", "-D", "--defined-only", nat.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\bT (accbpg_\w+)", nm))
    assert declared <= exported


def test_library_is_sm100a_with_dmma():
    from accbpg_and_fw_b200 import _native as nat
    out = subprocess.run(["cuobjdump", "-lelf", nat.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", "_ZN6accbpg16syrk_dmma_kernelILb1EEEvNS_10SyrkParamsE",
                           nat.LIB_PATH], capture_output=True, text=True).stdout
    assert sass.count("DMMA.8x8x4") >= 64 and "LDGSTS" in sass           # cp.async fallback mainloop
    tma = subprocess.run(["cuobjdump", "-sass", "-fun", "_ZN6accbpg15syrk_tma_kernelENS_10SyrkParamsE14CUtensorMap_stS1_",
                          nat.LIB_PATH], capture_output=True, text=True).stdout
    # TMA mainloop: tensor-map bulk loads signalled on mbarriers feed the FP64 tensor pipe
    assert tma.count("DMMA.8x8x4") >= 64 and "UTMALDG" in tma and "SYNCS" in tma


def test_frank_wolfe_persistent_loop_is_tma_fed():
    """The persistent Frank-Wolfe loop streams V with tensor copies (3-D and 2-D) signalled on mbarriers (UTMALDG +
    SYNCS) and releases / acquires its flag words at GPU scope."""
    from accbpg_and_fw_b200 import _native as nat
    sass = subprocess.run(["cuobjdump", "-sass", nat.LIB_PATH], capture_output=True, text=True).stdout
    funcs, cur = {}, None
    for line in sass.splitlines():
        if "Function :" in line:
            cur = line.split("Function :")[1].strip()
            funcs[cur] = []
        elif cur is not None:
            funcs[cur].append(line)

    def body(substr):
        hits = [k for k in funcs if substr in k]
        assert hits, substr
        return "\n".join(funcs[hits[0]])

    b = body("fw_persist_ring_kernel")
    assert "UTMALDG.3D" in b and "UTMALDG.2D" in b and "SYNCS" in b
    assert re.search(r"ST\w*\.E\.64\.STRONG\.GPU", b) and re.search(r"LD\w*\.E\.64\.STRONG\.GPU", b)


def test_peer_memory_kernels_use_system_scope_release_acquire():
    """The NVLink peer-memory exchanges rest on: payload stores, a system-scope fence, a release store of the flag word;
    an acquire load of the flag (which also drops stale L1 lines) before the payload is read.  Check that this is what
    was compiled: MEMBAR.*.SYS + STG.*.STRONG.SYS on the sending side, LDG.*.STRONG.SYS + CCTL.IVALL on the waiting side."""
    from accbpg_and_fw_b200 import _native as nat
    sass = subprocess.run(["cuobjdump", "-sass", nat.LIB_PATH], capture_output=True, text=True).stdout
    funcs = {}
    cur = None
    for line in sass.splitlines():
        if "Function :" in line:
            cur = line.split("Function :")[1].strip()
            funcs[cur] = []
        elif cur is not None:
            funcs[cur].append(line)

    def body(substr):
        hits = [k for k in funcs if substr in k]
        assert hits, substr
        return "\n".join(funcs[hits[0]])

    for sender in ("syrk_reduce_push_kernel", "burg_prepare_push_kernel", "peer_vec_push_kernel",
                   "peer_sum_scalars_kernel", "peer_argmin_pair_kernel", "fw_pass_kernel", "fw_decide_peer_kernel"):
        b = body(sender)
        assert re.search(r"MEMBAR\.\w+\.SYS", b) and re.search(r"STG\.E\.64\.STRONG\.SYS", b), sender
    for waiter in ("gram_sum_received_kernel", "peer_wait_kernel", "peer_vec_sum_kernel", "peer_sum_scalars_kernel",
                   "peer_argmin_pair_kernel", "fw_decide_peer_kernel", "fw_hv_kernel"):
        b = body(waiter)
        assert re.search(r"LDG\.E\.64\.STRONG\.SYS", b) and "CCTL.IVALL" in b and "NANOSLEEP" in b, waiter


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import accbpg_and_fw_b200 as acc
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        acc.D_opt_design(8, 20, randseed=1)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "accbpg_and_fw_b200")
    pat = re.compile(r"^\s*(from\s+oracle\b|import\s+oracle\b|from\s+\.+oracle\b)|accbpg_oracle|importlib.*oracle|"
                     r"oracle[/\\]", re.M)
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, fn)).read()
                assert not pat.search(text), f"{fn} reaches into the oracle package"


def test_solve_theta_matches_oracle():
    from accbpg_and_fw_b200.drivers import solve_theta
    for theta in (1.0, 0.5, 0.0123):
        for gamma in (1.0, 1.5, 2.0, 3.0):
            for ratio in (1, 0.8, 1.2):
                assert solve_theta(theta, gamma, ratio) == orc.solve_theta(theta, gamma, ratio)


def test_column_partition():
    from accbpg_and_fw_b200.dist import ColumnShard
    for n in (1, 2, 7, 200, 50001, 1000000):
        for world in (1, 2, 3, 4, 8):
            offs = ColumnShard.partition(n, world)
            assert offs[0] == 0 and offs[-1] == n and len(offs) == world + 1
            assert all(b >= a for a, b in zip(offs, offs[1:]))
            assert all(o % 2 == 0 for o in offs[:-1])
            sizes = [b - a for a, b in zip(offs, offs[1:])]
            assert max(sizes) - min(sizes) <= 3
    sh = ColumnShard(10, rank=1, world=2)
    assert (sh.lo, sh.hi, sh.n_local) == (6, 10, 4) or (sh.lo, sh.hi) == (4, 10) or sh.lo % 2 == 0
    assert sh.owner(0) == 0 and sh.owner(9) == 1


def test_libsvm_parser_matches_reference_matrix(golden_ops):
    from accbpg_and_fw_b200.problems import load_libsvm_dense
    X, y = load_libsvm_dense(os.path.join(GOLDEN, "housing_libsvm.txt"))
    assert X.shape == (506, 13) and y.shape == (506,)
    assert np.array_equal(np.ascontiguousarray(X.T), golden_ops["housing_H"])


def test_libsvm_parser_edge_cases(tmp_path):
    from accbpg_and_fw_b200.problems import load_libsvm_dense
    p = tmp_path / "t.txt"
    p.write_text("# comment only\n1.5 1:2.0 3:4.0 # trailing\n\n-1 2:1e-3\n")
    X, y = load_libsvm_dense(str(p))
    assert X.tolist() == [[2.0, 0.0, 4.0], [0.0, 1e-3, 0.0]] and y.tolist() == [1.5, -1.0]
    p.write_text("1 3:1 2:1\n")
    with pytest.raises(ValueError):
        load_libsvm_dense(str(p))


_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[3])
from accbpg_and_fw_b200.dist import ColumnShard
rank, world = int(sys.argv[1]), 2
os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = sys.argv[2]
dist.init_process_group("gloo", rank=rank, world_size=world)
sh = ColumnShard(11)
full = torch.arange(11, dtype=torch.float64) * 1.5
loc = sh.part(full)
assert torch.equal(sh.gather(loc), full)
t = torch.tensor([float(loc.sum())], dtype=torch.float64); sh.sum_(t); assert t.item() == full.sum().item()
# argmin with an exact tie across ranks: value 0.25 at global columns 3 (rank 0) and 8 (rank 1) -> 3 wins
g = torch.ones(11, dtype=torch.float64); g[3] = 0.25; g[8] = 0.25
gl = sh.part(g)
li = int(torch.argmin(gl)); pair = torch.tensor([float(gl[li]), float(li + sh.lo)], dtype=torch.float64)
sh.argmin_(pair); assert pair.tolist() == [0.25, 3.0], pair
m = torch.tensor([float(gl.min())], dtype=torch.float64); sh.min_(m); assert m.item() == 0.25
assert sh.owner(3) == 0 and sh.owner(8) == 1
# equal-length gather used by the sharded Burg-simplex root-find and the FW selection records: padding = +inf
pad = torch.full((sh.width,), float("inf"), dtype=torch.float64); pad[: loc.numel()] = loc
allv = torch.empty(sh.width * world, dtype=torch.float64); sh.all_gather_equal(allv, pad)
got = torch.cat([allv[r * sh.width: r * sh.width + (sh.offsets[r + 1] - sh.offsets[r])] for r in range(world)])
assert torch.equal(got, full) and torch.isinf(allv).sum().item() == sh.width * world - 11
# the NVLink peer-memory exchanges need NCCL: on any other backend the buffer factory declines and callers use the
# collectives above
from accbpg_and_fw_b200.dist import peer_buffers
assert peer_buffers(sh, torch.device("cpu"), [(16, torch.float64), (2, torch.int64)]) is None
assert peer_buffers(None, torch.device("cpu"), [(16, torch.float64)]) is None
# ... and so does the scalar exchange that also carries the status words (drivers then use all-reduce sum + max)
assert sh.sum_scalars_into(t, t) is False
dist.destroy_process_group()
print("ok", rank)
'''


def test_column_shard_collectives_gloo_world2(tmp_path):
    """World-size-2 gloo run of the sharding collectives (sum, min, gather, lowest-index argmin)."""
    script = tmp_path / "w.py"
    script.write_text(_WORKER)
    port = str(29500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), str(r), port, ROOT], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"ok {r}" in o, o


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs next to the GPU arm) prints one JSON line with the
    contract's keys; no GPU is touched."""
    import json
    import sys
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "abpg_gamma2_iterations_per_sec"
    for key in ("value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype",
                "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    from oracle import ref_loader
    assert line["cpu_baseline"]["kind"] == ("reference" if ref_loader.locate() else "port")
    assert line["cpu_baseline"]["cores"] == (os.cpu_count() or 1)      # set explicitly, whatever the launcher exported
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"] > 0


@pytest.mark.parametrize("name", ["housing", "abalone", "bodyfat", "mpg"])
def test_libsvm_sparse_loader_matches_dense(name):
    """The compressed-column form of H = X^T (one column per sample, file order) densifies to exactly what the dense
    loader builds (which the reference's own loader + .toarray('C') reproduces bit for bit, test_oracle_golden.py)."""
    import scipy.sparse as sp
    from accbpg_and_fw_b200.problems import load_libsvm_dense, load_libsvm_sparse
    path = os.path.join(GOLDEN, name + "_libsvm.txt")
    X, y = load_libsvm_dense(path)
    indptr, indices, values, nfeat, y2 = load_libsvm_sparse(path)
    assert indptr.dtype == np.int64 and indices.dtype == np.int32 and nfeat == X.shape[1] and np.array_equal(y, y2)
    H = sp.csc_matrix((values, indices, indptr), shape=(nfeat, indptr.size - 1)).toarray()
    assert np.array_equal(H, X.T)
    assert np.all(np.diff(indptr) >= 0) and indptr[-1] == values.size
