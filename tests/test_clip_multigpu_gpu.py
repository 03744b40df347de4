"""A whole clip on several GPUs: tools/clip_check.py under torch.distributed.run compares the VAE encode / decode split by frame over
the ranks with the single-GPU stages (bit-identical per frame, within 0.03 std batched) and a 3-step image_guided_synthesis under
parallel.shard_model with the single-GPU call (within 0.15).  The NCCL cases need >= 2 CUDA devices (4 for world 4); the shared-GPU
case runs two ranks on one device over gloo."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1200)]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("world,peer", [(2, "1"), (2, "0"), (4, "1"), (4, "0")])
def test_clip_sharded_matches_single_gpu(world, peer):
    """world 2: CFG split (the U-Net exchanges no frames), VAE frames 13 / 12; world 4: 2 x 2, VAE frames 7 / 6 / 6 / 6.
    peer selects the U-Net's frame exchange (NVLink peer-memory kernels or NCCL); the VAE gathers use NCCL either way."""
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} CUDA devices")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(ROOT, "tools", "clip_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1100, env=dict(os.environ, VC_PEER_COMM=peer))
    print(r.stdout[-4000:], r.stderr[-2000:])
    assert r.returncode == 0 and "CLIP_CHECK_OK" in r.stdout


def test_clip_two_ranks_on_one_gpu():
    """World 2 (CFG split) with both ranks on cuda:0 over gloo: the sharded VAE stages and the split denoise loop on the real kernels on a
    box with a single GPU."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29542", os.path.join(ROOT, "tools", "clip_check.py"), "--shared-gpu"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1100)
    print(r.stdout[-4000:], r.stderr[-2000:])
    assert r.returncode == 0 and "CLIP_CHECK_OK" in r.stdout
