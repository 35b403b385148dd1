"""Where the data-parallel step spends its extra time (VERDICT r1 item 6): per-bucket all-reduce durations on the comm stream and
the exposed tail between the end of backward and the start of the SGD pass, eager launches, CUDA events, max over ranks.
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29544 profiles/dp_bucket_times.py"""
import copy, ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, torch.distributed as dist
import hpfg_b200 as hb
from hpfg_b200 import _lib as L
from hpfg_b200.losses import ssl_loss_raw

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
torch.manual_seed(1337)
student = hb.UNet(1, 4, precision="bf16").to(dev)
teacher = copy.deepcopy(student)
step = hb.MeanTeacherStep(student, teacher)
g = torch.Generator().manual_seed(1337 + rank)
x = torch.rand(32, 1, 224, 224, generator=g).to(dev)
y = torch.randint(0, 4, (8, 224, 224), generator=g).to(dev)
for _ in range(5):
    step.step(x, y)
torch.cuda.synchronize()
dist.barrier()
ev = lambda: torch.cuda.Event(enable_timing=True)
reps = 20
acc = {}
lib = L.lib()
buckets = hb.gradient_buckets(1, 4)
for _ in range(reps):
    step._next_iteration()
    main = torch.cuda.current_stream(dev)
    side = step._side_stream(dev)
    shape = (32, 4, 224, 224)
    e_start, e_bwd0, e_bwd1, e_sgd0, e_sgd1 = ev(), ev(), ev(), ev(), ev()
    e_start.record(main)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        _, t_out = step._forward(teacher, x, False, step._persistent("t_out", shape, dev), None)
    plan, out = step._forward(student, x, True, step._persistent("s_out", shape, dev), None)
    main.wait_stream(side)
    r = ssl_loss_raw(L.LOSS_MT, out, t_out[8:], y, 8, cons_weight=0.001)
    e_bwd0.record(main)
    L.check(lib.hpfg_unet_backward(plan.handle, L.ptr(student.flat_params), L.ptr(r["dstudent"]), L.ptr(step.grads), 0, L.stream_ptr(dev)))
    e_bwd1.record(main)
    if step._comm is None:
        step._comm = torch.cuda.Stream(device=dev)
    comm = step._comm
    evs = []
    for b, (off, cnt) in enumerate(buckets):
        L.check(lib.hpfg_unet_bucket_wait(plan.handle, b, ctypes.c_void_p(comm.cuda_stream)))
        with torch.cuda.stream(comm):
            a, z = ev(), ev()
            a.record(comm)
            dist.all_reduce(step.grads[off:off + cnt])
            z.record(comm)
            evs.append((a, z))
    main.wait_stream(comm)
    e_sgd0.record(main)
    step._opt_step(step._trained[0], None, teacher)
    e_sgd1.record(main)
    torch.cuda.synchronize()
    vals = {"forward+loss": e_start.elapsed_time(e_bwd0), "backward (main stream)": e_bwd0.elapsed_time(e_bwd1),
            "exposed tail: backward end -> SGD start": e_bwd1.elapsed_time(e_sgd0), "sgd+ema": e_sgd0.elapsed_time(e_sgd1),
            "whole step": e_start.elapsed_time(e_sgd1)}
    for b, (a, z) in enumerate(evs):
        vals["bucket %d all-reduce (%d params)" % (b, buckets[b][1])] = a.elapsed_time(z)
        vals["bucket %d end relative to backward end" % b] = e_bwd1.elapsed_time(z)
    for k, v in vals.items():
        acc[k] = acc.get(k, 0.0) + v / reps
keys = list(acc)
t = torch.tensor([acc[k] for k in keys], device=dev)
dist.all_reduce(t, op=dist.ReduceOp.MAX)
if rank == 0:
    print("data-parallel Mean-Teacher step on %d GPUs, eager launches, ms (max over ranks, mean of %d steps)" % (world, reps))
    for k, v in zip(keys, t.tolist()):
        print("  %-48s %8.3f" % (k, v))
dist.barrier()
dist.destroy_process_group()
