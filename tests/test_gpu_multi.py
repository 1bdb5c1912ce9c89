"""Several GPUs, one stream (csrc/dist.cpp): the library shards the master blocks over the GPUs of the
box, NCCL scatters the byte ranges and gathers the compressed bits at their final bit offsets.  The
result must be the reference's bytes -- the same bytes one GPU produces.  Skipped with fewer GPUs than a case
needs; the reference's answers are looked up before that."""
import os
import subprocess
import sys
import tempfile

import pytest

from zopfli_b200 import corpus

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ngpus():
    import torch
    return torch.cuda.device_count()


CODE = ("import sys; sys.path.insert(0, %r); import zopfli_b200 as zb; d = open(sys.argv[1], 'rb').read(); "
        "fmt = int(sys.argv[3]); it = int(sys.argv[4]); "
        "open(sys.argv[2], 'wb').write(zb.compress(d, fmt, numiterations=it))" % ROOT)


@pytest.mark.parametrize("ngpus", [2, 3, 4, 8])
def test_one_process_several_gpus_equals_reference(ref, ngpus):
    """ZopfliCompress with ZOPFLI_B200_GPUS=N (ncclCommInitAll, one host thread per GPU)."""
    cases = [(corpus.synth_text(5300000, 2), 0, 2),              # 6 master blocks, ragged tail, gzip
             (corpus.synth_text(2000001, 3), 1, 1),              # fewer master blocks than ranks at N >= 4; zlib
             (corpus.synth_binary(3100000, 4) + corpus.random_bytes(1200000), 2, 1)]  # stored blocks cross rank boundaries
    want = [ref.compress(data, fmt, numiterations=it) for data, fmt, it in cases]
    if _ngpus() < ngpus:
        pytest.skip("needs %d GPUs" % ngpus)
    with tempfile.TemporaryDirectory() as td:
        for i, (data, fmt, it) in enumerate(cases):
            src, out = os.path.join(td, "in%d" % i), os.path.join(td, "out%d" % i)
            open(src, "wb").write(data)
            subprocess.check_call([sys.executable, "-c", CODE, src, out, str(fmt), str(it)],
                                  env=dict(os.environ, ZOPFLI_B200_GPUS=str(ngpus)))
            assert open(out, "rb").read() == want[i], (ngpus, i)


def test_one_process_per_gpu_under_torchrun(ref):
    """ZopfliB200DistInit + ZopfliB200DistCompress, the id broadcast through torch.distributed."""
    data = corpus.synth_text(4200000, 5)
    want = ref.compress(data, 0, numiterations=2)
    n = min(_ngpus(), 4)
    if n < 2:
        pytest.skip("needs 2 GPUs")
    with tempfile.TemporaryDirectory() as td:
        src, out = os.path.join(td, "in"), os.path.join(td, "out")
        open(src, "wb").write(data)
        script = os.path.join(td, "w.py")
        open(script, "w").write('''
import os, sys
sys.path.insert(0, %r)
import numpy as np, torch, torch.distributed as dist
import zopfli_b200 as zb
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
lib = zb.library()
idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
if rank == 0:
    idt.copy_(torch.frombuffer(bytearray(lib.dist_unique_id()), dtype=torch.uint8))
dist.broadcast(idt, 0)
lib.dist_init(rank, world, idt.cpu().numpy().tobytes())
data = open(sys.argv[1], "rb").read()
host = np.frombuffer(data, dtype=np.uint8).copy() if rank == 0 else np.zeros(1, np.uint8)
for staged in (False, True):
    ob = lib.dist_compress_ptr_nocopy(host.ctypes.data, len(data), zb.ZOPFLI_FORMAT_GZIP, staged=staged, numiterations=2)
    if rank == 0:
        open(sys.argv[2] + str(int(staged)), "wb").write(ob.tobytes())
        ob.close()
dist.barrier()
lib.dist_finalize()
dist.destroy_process_group()
''' % ROOT)
        subprocess.check_call([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
                               "--master-addr", "127.0.0.1", "--master-port", "29611", script, src, out],
                              env=dict(os.environ, NCCL_DEBUG="WARN"))
        assert open(out + "0", "rb").read() == want
        assert open(out + "1", "rb").read() == want
