"""One rank of the two-rank training-metrics test (tests/test_gpu_train_metrics.py), launched by
torch.distributed.run: Trainer.fit over this rank's shard of a replay, with the values each step logged on this rank
read after the step.  Each rank writes its recorded rows and logged values to argv[1]/rank<r>.json."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402


def main(out_dir):
    from tacorl_b200 import runtime
    from tacorl_b200 import trainer as TR
    from tacorl_b200.replay import DeviceReplay, ReplayIndex
    from tests.test_gpu_validation import _episodes, _module
    rank, world, local = (int(os.environ[k]) for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
    torch.cuda.set_device(local)
    index = ReplayIndex(_episodes({"rgb_static": (84, 84)}, seed=12, lengths=[14, 9, 30, 6, 11]), rank=rank,
                        world_size=world)
    train = DeviceReplay(index, 3, kind="play_lmp", min_window=4, max_window=8, pad=4, seed=3,
                         device=torch.device("cuda", local))
    m = _module("play_lmp")
    logged = []
    orig = runtime.TrainMetricsRecorder.step_done

    def step_done(self, global_step, epoch):
        torch.cuda.synchronize()
        logged.append({k: v.float().item() for k, v in m.logged.items() if k.startswith("train/")})
        orig(self, global_step, epoch)
    runtime.TrainMetricsRecorder.step_done = step_done
    torch.manual_seed(1)
    tr = TR.Trainer(max_steps=6, precision="fp32", steps_per_epoch=3, log_every_n_steps=2)
    tr.fit(m, train)
    h = tr.train_history
    with open(os.path.join(out_dir, f"rank{rank}.json"), "w") as f:
        json.dump({"keys": h.keys, "steps": h.steps.tolist(), "rows": h.values.tolist(),
                   "logged": [[row[k] for k in h.keys] for row in logged],
                   "epoch_metrics": tr.train_epoch_metrics}, f)
    torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1])
