"""One rank of the two-rank validation test (tests/test_gpu_validation.py), launched by torch.distributed.run:
Trainer.validate over this rank's shard of a split whose shards hold different item counts.  Rank 0 writes the
global metrics and the item count of each shard to argv[1]."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402


def episodes():
    from tests.test_gpu_validation import _episodes
    return _episodes({"rgb_static": (84, 84)}, seed=12, lengths=[14, 9, 30, 6, 11])


def shard_replay(index, device):
    from tacorl_b200.replay import DeviceReplay
    return DeviceReplay(index, 5, kind="play_lmp", min_window=4, max_window=8, seed=11, device=device, mode="sweep")


def main(out):
    from tacorl_b200 import trainer as TR
    from tacorl_b200.replay import ReplayIndex
    from tests.test_gpu_validation import _module
    rank, world, local = (int(os.environ[k]) for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
    torch.cuda.set_device(local)
    val = shard_replay(ReplayIndex(episodes(), rank=rank, world_size=world), torch.device("cuda", local))
    [metrics] = TR.Trainer(precision="fp32").validate(_module("play_lmp"), val)
    if rank == 0:
        items = [len(ReplayIndex(episodes(), rank=r, world_size=world).items("play_lmp", 4)) for r in range(world)]
        with open(out, "w") as f:
            json.dump({"metrics": metrics, "items": items}, f)
    torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1])
