"""python tools/train_bench.py [C2 C3 C4]   (single GPU) -- or under torchrun for N GPUs."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, torch.distributed as dist
from mog_asr_b200.air import bench_train

world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
dev = torch.device("cuda", local); torch.cuda.set_device(dev)
pg = None
if world > 1:
    dist.init_process_group("nccl", device_id=dev); pg = dist.group.WORLD
names = [a for a in sys.argv[1:] if a in bench_train.CONFIGS] or ["C2", "C3", "C4"]
for n in names:
    for fixed, graph, ref_trips in ((False, False, False), (True, False, False), (True, True, False), (True, True, True)):
        r = bench_train.run(n, dev, steps=20, warmup=5, process_group=pg, always_max_steps=fixed, graph=graph,
                            reference_trip_count=ref_trips)
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps(r), flush=True)
if world > 1:
    dist.destroy_process_group()
