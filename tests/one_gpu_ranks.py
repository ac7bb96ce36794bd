"""torchrun entry point of the sharded-tool tests on a box with one GPU: runs ``tools.opt_arti`` with every rank
on cuda:0 and the process group over gloo, since NCCL refuses two ranks on one device.  Everything else (the
barrier around ``--synthetic``, sharding, per-rank outputs, rank 0's AP table, the reduced summary line) is the
tool's own distributed path."""
import os
import sys

import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from articulation3d_b200.tools import opt_arti  # noqa: E402

_init = dist.init_process_group


def _gloo(backend=None, *args, device_id=None, **kwargs):
    return _init("gloo", *args, **kwargs)


os.environ["LOCAL_RANK"] = "0"
dist.init_process_group = _gloo
opt_arti.main(sys.argv[1:])
