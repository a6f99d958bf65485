"""N ranks, ONE PROCESS PER RANK (CUDA-IPC peers, the fused peer stores of the pair kernel on - the configuration
bench.py runs), against the single-rank run: bit-identical state, diagnostics and interaction counters after three
full loop bodies with accretion and bounds removals.

Two collective backends carry the same engine code:
  * host  - shared-memory collectives (sph_comm_init_host); the ranks share cuda:0, so these cases run on the 1-GPU box;
  * nccl  - the production backend, one GPU per rank; skipped when fewer GPUs than ranks are visible.
"""
import os
import subprocess
import sys
import uuid

import numpy as np
import pytest

from summersph_b200 import MODE_VARIABLE_H, MODE_FIXED_H

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
WORKER = os.path.join(HERE, "_mp_rank.py")


def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def run_ranks(tmp_path, tag, world, comm, mode, steps=3, env_extra=None, n=60_000, domains=0, extra="-", ics="-", case="-"):
    """Launch `world` worker processes; returns the list of result dicts (one per rank)."""
    token = ""
    if world > 1:
        if comm == "nccl":
            from summersph_b200.engine import Engine, load_library
            import ctypes as C
            buf = (C.c_char * 128)()
            assert load_library().sph_comm_unique_id(buf) == 0
            token = bytes(buf).hex()
        else:
            token = "/sphb200_" + uuid.uuid4().hex[:16]
    env = dict(os.environ)
    env.update(env_extra or {})
    procs, outs = [], []
    for r in range(world):
        out = str(tmp_path / f"{tag}_r{r}.npz")
        dev = r if comm == "nccl" else 0
        outs.append(out)
        procs.append(subprocess.Popen([sys.executable, WORKER, str(r), str(world), comm, str(dev), str(mode), str(steps), out, token or "-", str(n), str(domains), extra, ics, case],
                                      env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    logs = []
    for p in procs:
        try:
            o, _ = p.communicate(timeout=float(os.environ.get('SPH_TEST_RANK_TIMEOUT', '900')))
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise
        logs.append(o)
    for r, p in enumerate(procs):
        assert p.returncode == 0, f"rank {r} failed:\n{logs[r][-4000:]}"
    return [dict(np.load(o)) for o in outs]


def assert_identical(res, ref, what):
    for k in ref:
        assert k in res, (what, k)
        a, b = res[k], ref[k]
        assert a.shape == b.shape, (what, k, a.shape, b.shape)
        assert np.array_equal(a, b, equal_nan=True), (what, k, float(np.nanmax(np.abs(a - b))) if a.dtype.kind == "f" else "int")


@pytest.fixture(scope="module")
def single_rank(tmp_path_factory, built_engine):
    d = tmp_path_factory.mktemp("one_rank")
    return {m: run_ranks(d, f"one{m}", 1, "host", m)[0] for m in (MODE_VARIABLE_H, MODE_FIXED_H)}


def test_replicated_far_reuse_bit_identical(built_engine, tmp_path):
    """A case that removes nothing: evaluation A of steps 2.. keeps evaluation B's far-field gravity and adds the recorded
    near pairs.  The gravity runs - and with them the recorded pairs and their order - are the same for any rank count,
    so the replicated form stays bit-identical to one rank."""
    env = {"SPH_TEST_QUIET": "1"}
    ref = run_ranks(tmp_path, "q1", 1, "host", MODE_VARIABLE_H, steps=4, env_extra=env, n=30_000)[0]
    assert int(ref["far_reuse"][0]) >= 2
    res = run_ranks(tmp_path, "q2", 2, "host", MODE_VARIABLE_H, steps=4, env_extra=env, n=30_000)
    for r in range(2):
        assert_identical(res[r], ref, f"quiet rank {r}")


@pytest.mark.parametrize("mode", [MODE_VARIABLE_H, MODE_FIXED_H])
@pytest.mark.parametrize("world,env", [(2, {}), (3, {}), (2, {"SPH_B200_NO_FUSED_PUSH": "1"})])
def test_process_per_rank_shared_gpu_bit_identical(mode, world, env, single_rank, tmp_path):
    """Virtual ranks: every rank is its own process on cuda:0 (CUDA IPC between them, host-segment collectives)."""
    res = run_ranks(tmp_path, f"h{world}", world, "host", mode, env_extra=env)
    for r in range(world):
        assert_identical(res[r], single_rank[mode], f"world {world} rank {r} {env}")


@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("mode", [MODE_VARIABLE_H, MODE_FIXED_H])
@pytest.mark.parametrize("env", [{}, {"SPH_B200_NO_FUSED_PUSH": "1"}, {"SPH_B200_NO_P2P": "1"}])
def test_process_per_gpu_nccl_bit_identical(mode, env, single_rank, tmp_path):
    """The production configuration: one process per GPU, NCCL collectives, CUDA-IPC peers, fused PeerOut stores
    (and the two developer fallbacks: copy-engine exchange, NCCL broadcasts)."""
    res = run_ranks(tmp_path, "n2", 2, "nccl", mode, env_extra=env)
    for r in range(2):
        assert_identical(res[r], single_rank[mode], f"nccl rank {r} {env}")


@pytest.mark.skipif(_ngpu() < 4, reason="needs 4 GPUs")
def test_four_gpus_nccl_bit_identical(single_rank, tmp_path):
    res = run_ranks(tmp_path, "n4", 4, "nccl", MODE_VARIABLE_H)
    for r in range(4):
        assert_identical(res[r], single_rank[MODE_VARIABLE_H], f"nccl4 rank {r}")
