"""SP+LP training benchmark: the spatial stage(s) of ResNet / AmoebaNet-D run on image tiles across
P GPUs (halo exchange inside conv_spatial / Pool), the remaining pipeline stages on one GPU each.

Same command line as the reference's benchmarks/spatial_parallelism/benchmark_{resnet,amoebanet}_sp.py
(torchgems.parser flags), launched with torchrun instead of mpirun_rsh:

    torchrun --nnodes=1 --nproc-per-node 5 --master-addr 127.0.0.1 \\
        benchmarks/spatial_parallelism/benchmark_amoebanet_sp.py --image-size 1024 --num-spatial-parts 4 \\
        --slice-method square --split-size 2 --batch-size 1 --num-layers 18 --num-filters 416 --dtype bf16

world size = spatial_size * P + split_size - spatial_size.  Extra flags of this script: --dtype
{fp32,bf16} (bf16 puts the spatial convs on the tcgen05 kernels), --steps N (synthetic batches per
epoch, default 10).  APP 3 (synthetic) needs no dataset; APP 1/2 use torchvision like the reference.
"""
import math
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))

from mpi4dl_b200.torchgems import comm as gems_comm  # noqa: E402
from mpi4dl_b200.torchgems import parser  # noqa: E402
from mpi4dl_b200.torchgems.mp_pipeline import model_generator  # noqa: E402
from mpi4dl_b200.torchgems.train_spatial import (get_shapes_spatial, split_input, train_model_spatial,  # noqa: E402
                                                 verify_spatial_config)
from mpi4dl_b200.torchgems.utils import get_depth  # noqa: E402


def _builders(kind, args, mb, image_size, spatial_kw):
    """(sequential model at the small tracing size, its size, spatial model at the real size)."""
    if kind == "resnet":
        from mpi4dl_b200.models import resnet, resnet_spatial
        seq_size, depth = 32, get_depth(2, 12)
        seq = resnet.get_resnet_v2((mb, 3, seq_size, seq_size), depth=depth, num_classes=args.num_classes)
        if args.halo_d2:      # fused-halo cells (benchmark_resnet_sp.py:183-195): the builder also returns the balance it adjusted
            from mpi4dl_b200.models import resnet_spatial_d2
            model, new_balance = resnet_spatial_d2.get_resnet_v2(depth=depth, num_classes=args.num_classes,
                                                                 fused_layers=args.fused_layers, **spatial_kw)
            spatial_kw["balance_out"] = new_balance
            return seq, seq_size, model
        model = resnet_spatial.get_resnet_v2(depth=depth, num_classes=args.num_classes, fused_layers=args.fused_layers,
                                             **spatial_kw)
        return seq, seq_size, model
    from mpi4dl_b200.models import amoebanet
    if args.halo_d2:                       # fused-halo cells: two wide exchanges per normal cell, valid convs after
        from mpi4dl_b200.models import amoebanet_d2 as spatial_builder
    else:
        spatial_builder = amoebanet
    seq_size = min(512, image_size)
    seq = amoebanet.amoebanetd(num_classes=args.num_classes, num_layers=args.num_layers, num_filters=args.num_filters)
    kw = dict(spatial_kw)
    kw.pop("input_shape", None)
    model = spatial_builder.amoebanetd_spatial(num_classes=args.num_classes, num_layers=args.num_layers,
                                               num_filters=args.num_filters, **kw)
    return seq, seq_size, model


def _batches(args, image_size, batch_size, steps):
    """Yield (images, labels) host batches."""
    if args.app == 3:
        g = torch.Generator().manual_seed(0)
        x = torch.randn(batch_size, 3, image_size, image_size, generator=g)
        y = torch.randint(0, args.num_classes, (batch_size,), generator=g)
        if torch.cuda.is_available():
            x, y = x.pin_memory(), y.pin_memory()
        for _ in range(steps):
            yield x, y
        return
    import torchvision
    import torchvision.transforms as transforms
    tf = transforms.Compose([transforms.ToTensor(), transforms.Normalize((0.5, 0.5, 0.5), (0.5, 0.5, 0.5))])
    torch.manual_seed(0)
    if args.app == 1:
        ds = torchvision.datasets.ImageFolder(args.datapath, transform=tf)
    else:
        ds = torchvision.datasets.CIFAR10(root=args.datapath, train=True, download=False, transform=tf)
    dl = torch.utils.data.DataLoader(ds, batch_size=batch_size * args.times, shuffle=(args.app == 1),
                                     num_workers=args.num_workers, pin_memory=True, drop_last=True)
    yield from dl


def main(kind):
    p = parser.get_parser()
    p.add_argument("--dtype", choices=["fp32", "bf16", "tf32"], default="fp32",
                   help="tf32: fp32 tensors, convolutions on the tensor cores with TF32 operands")
    p.add_argument("--steps", type=int, default=10)
    args = p.parse_args()
    gems_comm.initialize_cuda()
    np.random.seed(seed=1405)

    batch_size, parts, image_size = args.batch_size, args.parts, int(args.image_size)
    split_size, spatial_size, slice_method = args.split_size, args.spatial_size, args.slice_method
    nsp = [int(v) for v in args.num_spatial_parts.split(",")]
    num_spatial_parts = nsp[0] if len(nsp) == 1 else nsp
    P = nsp[0]
    balance = [int(v) for v in args.balance.split(",")] if args.balance else None
    if args.local_DP != 1:
        raise NotImplementedError("--local-DP > 1 is not built yet")
    verify_spatial_config(slice_method, image_size, nsp)

    mpi_comm = gems_comm.MPIComm(split_size=split_size, ENABLE_MASTER=False, ENABLE_SPATIAL=True,
                                 num_spatial_parts=num_spatial_parts, spatial_size=spatial_size)
    sync_allreduce = gems_comm.SyncAllreduce(mpi_comm)
    local_rank, split_rank = mpi_comm.rank, mpi_comm.split_rank
    mb = int(batch_size / parts)
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    if args.dtype == "tf32":
        from mpi4dl_b200.torchgems.spatial import set_fp32_math

        set_fp32_math("tf32")

    spatial_kw = dict(input_shape=(mb, 3, image_size, image_size), local_rank=local_rank % P, mp_size=split_size,
                      balance=balance, spatial_size=spatial_size, num_spatial_parts=num_spatial_parts, slice_method=slice_method)
    seq, seq_size, model = _builders(kind, args, mb, image_size, spatial_kw)
    # per-stage output shapes: traced on the small sequential model, scaled to the real image and tiling
    gen_seq = model_generator(model=seq, split_size=split_size, input_size=(mb, 3, seq_size, seq_size), balance=balance)
    gen_seq.get_output_shapes(GET_SHAPES_ON_CUDA=torch.cuda.is_available())
    shapes = get_shapes_spatial(gen_seq.shape_list, slice_method, spatial_size, nsp, int(image_size / seq_size))
    del seq, gen_seq

    # (the D2 ResNet builder inserts halo layers into stage 0 and hands back the balance that accounts for them)
    model_gen = model_generator(model=model.to(dtype), split_size=split_size, input_size=(mb, 3, image_size, image_size),
                                balance=spatial_kw.get("balance_out", balance), shape_list=shapes)
    model_gen.ready_model(split_rank=split_rank)
    del model
    trainer = train_model_spatial(model_gen, local_rank, batch_size, epochs=1, spatial_size=spatial_size,
                                  num_spatial_parts=num_spatial_parts, parts=parts, ASYNC=True, GEMS_INVERSE=False,
                                  slice_method=slice_method, mpi_comm=mpi_comm)
    sync_allreduce.sync_model_spatial(model_gen)
    is_tile = local_rank < spatial_size * P
    cuda = torch.cuda.is_available()

    perf = []
    for epoch in range(args.num_epochs):
        loss_sum = correct_sum = 0.0
        n = 0
        for inputs, labels in _batches(args, image_size, batch_size, args.steps):
            if cuda:
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
            else:
                w0 = time.perf_counter()
            x = split_input(inputs, image_size, slice_method, local_rank, nsp) if local_rank < P else inputs
            loss, correct = trainer.run_step(x, labels)
            if is_tile:
                sync_allreduce.apply_allreduce(model_gen, mpi_comm.spatial_allreduce_grp)
            trainer.update()
            if cuda:
                t1.record()
                torch.cuda.synchronize()
                dt = t0.elapsed_time(t1) / 1000
            else:
                dt = time.perf_counter() - w0
            loss_sum += loss
            correct_sum += correct
            n += 1
            if local_rank == 0:
                print("Epoch: %d images per sec:%s" % (epoch, batch_size / dt), flush=True)
                perf.append(batch_size / dt)
            if local_rank == mpi_comm.size - 1:
                print("Step :%d, LOSS: %s, Global loss: %s Acc: %s" % (n - 1, loss, loss_sum / n, correct), flush=True)
        if local_rank == mpi_comm.size - 1 and n:
            print("Epoch %d Global loss: %s Acc %s" % (epoch, loss_sum / n, correct_sum / n), flush=True)
    if local_rank == 0 and perf:
        print("Mean %s Median %s" % (sum(perf) / len(perf), np.median(perf)), flush=True)
    import torch.distributed as dist
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    kind = "resnet"
    if "--model" in sys.argv:
        i = sys.argv.index("--model")
        kind = sys.argv[i + 1]
        del sys.argv[i:i + 2]
    main(kind)
