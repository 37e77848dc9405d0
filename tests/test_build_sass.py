"""Static evidence, on the CPU, that the in-tree library is the sm_100a product the design describes: every embedded
cubin targets sm_100a, the rollout / forward tile kernels issue tcgen05 MMAs with tensor-memory loads and stores
(SASS UTCHMMA / LDTM / STTM, /opt/skills/guides/B200_PROFILING.md's mnemonic table), and the streaming world step moves
its tiles with bulk (TMA) copies in both directions (UBLKCP)."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def sass():
    import swarm_b200 as sb
    # cuobjdump ships beside nvcc, which the build also finds when the CUDA bin directory is not on PATH
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.path.dirname(sb._build._nvcc()), "cuobjdump")
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not found")
    lib = sb._build.build()
    elfs = subprocess.run([cuobjdump, "-lelf", lib], capture_output=True, text=True, check=True).stdout
    text = subprocess.run([cuobjdump, "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in text.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
        elif cur is not None:
            funcs[cur].append(line)
    return elfs, {k: "\n".join(v) for k, v in funcs.items()}


def test_every_cubin_targets_sm_100a(sass):
    elfs, _ = sass
    names = re.findall(r"ELF file\s+\d+:\s+(\S+)", elfs)
    assert names and all(n.endswith(".sm_100a.cubin") for n in names), names


def test_tile_kernels_use_tcgen05_and_tensor_memory(sass):
    _, funcs = sass
    # tile_kernel<MODE, TC, DENSE, FLOCK>: MODE 0 = rollout, 1 = forward; Lb1E as the second argument = tensor-core path
    tc = {k: v for k, v in funcs.items() if re.search(r"tile_kernelILi[01]ELb1E", k)}
    assert len(tc) >= 5, list(funcs)[:5]              # rollout x {3, 4 CTAs / SM} (+ Flocking variants), forward x 2
    for name, body in tc.items():
        assert "UTCHMMA" in body, f"{name}: no tcgen05.mma"
        assert "LDTM" in body and "STTM" in body, f"{name}: accumulators / A operand not in tensor memory"
        assert "UTCBAR" in body, f"{name}: no tcgen05.commit"
    ffma = [k for k in funcs if re.search(r"tile_kernelILi0ELb0E", k)]
    assert ffma and all("UTCHMMA" not in funcs[k] for k in ffma)       # the SWARM_TC=0 CUDA-core variant stays MMA-free


def test_streaming_world_step_uses_bulk_copies(sass):
    _, funcs = sass
    stream = {k: v for k, v in funcs.items() if "sim_step_stream_kernel" in k}
    assert len(stream) >= 4                            # EXTRAS x scenario
    for name, body in stream.items():
        assert "UBLKCP.S.G" in body and "UBLKCP.G.S" in body, f"{name}: no bulk loads / stores"
        assert "SYNCS" in body, f"{name}: no mbarrier wait"
