"""GEMS master + spatial parallelism: two replicas of the SP+LP pipeline on mirrored rank lines (replica
2's tiles live on the GPUs that hold replica 1's tail stages), each step trains --times batches
alternately through the two replicas, then the replicas' gradients are combined
(SyncAllreduce.apply_allreduce_master_master) -- or shipped rank <-> mirror around each half step with
--enable-master-comm-opt (train_spatial_model_master.run_step_allreduce).  Flags of the reference's
benchmarks/gems_master_with_spatial_parallelism scripts; torchrun launch:

    torchrun --nproc-per-node 8 benchmarks/gems_master_with_spatial_parallelism/benchmark_amoebanet_gems_master_with_sp.py \\
        --split-size 5 --num-spatial-parts 4 --slice-method square --image-size 1024 --batch-size 1 --times 2 \\
        --num-layers 18 --num-filters 416 --dtype bf16

world = spatial_size * P + split_size - spatial_size, and it must be >= 2 * P (verify_spatial_master_config).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.join(HERE, "..", ".."), os.path.join(HERE, ".."), os.path.join(HERE, "..", "spatial_parallelism")]

import common  # noqa: E402
from benchmark_sp import _builders  # noqa: E402
from mpi4dl_b200.torchgems import comm as gems_comm  # noqa: E402
from mpi4dl_b200.torchgems import parser  # noqa: E402
from mpi4dl_b200.torchgems.mp_pipeline import model_generator  # noqa: E402
from mpi4dl_b200.torchgems.train_spatial import get_shapes_spatial, split_input  # noqa: E402
from mpi4dl_b200.torchgems.train_spatial_master import train_spatial_model_master, verify_spatial_master_config  # noqa: E402


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
    times = max(2, args.times)
    nsp = [int(v) for v in args.num_spatial_parts.split(",")]
    num_spatial_parts = nsp[0] if len(nsp) == 1 else nsp
    P = nsp[0]
    balance = [int(v) for v in args.balance.split(",")] if args.balance else None
    if args.halo_d2 and kind == "resnet":
        raise NotImplementedError("--halo-D2 is built for AmoebaNet only")
    if args.local_DP != 1:
        raise NotImplementedError("--local-DP > 1 is not built")
    mb = int(batch_size / parts)
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    if args.dtype == "tf32":
        from mpi4dl_b200.torchgems.spatial import set_fp32_math

        set_fp32_math("tf32")

    comm1 = gems_comm.MPIComm(split_size=split_size, ENABLE_MASTER=False, ENABLE_SPATIAL=True,
                              num_spatial_parts=num_spatial_parts, spatial_size=spatial_size, LOCAL_DP_LP=1)
    verify_spatial_master_config(slice_method, image_size, nsp, spatial_size, comm1.mp_size)
    comm2 = gems_comm.MPIComm(split_size=split_size, ENABLE_MASTER=True, ENABLE_SPATIAL=True,
                              num_spatial_parts=num_spatial_parts, spatial_size=spatial_size, LOCAL_DP_LP=1,
                              DISABLE_INIT=True)
    gems_comm.sync_comms_for_master(comm1, comm2)

    gens, shapes = [], None
    for comm in (comm1, comm2):
        kw = dict(input_shape=(mb, 3, image_size, image_size), local_rank=comm.local_rank % comm.total_spatial_processes,
                  mp_size=split_size, balance=balance, spatial_size=spatial_size, num_spatial_parts=num_spatial_parts,
                  slice_method=slice_method)
        seq, seq_size, model = _builders(kind, args, mb, image_size, kw)
        if shapes is None:
            gen_seq = model_generator(model=seq, split_size=split_size, input_size=(mb, 3, seq_size, seq_size), balance=balance)
            gen_seq.get_output_shapes(GET_SHAPES_ON_CUDA=torch.cuda.is_available())
            shapes = get_shapes_spatial(gen_seq.shape_list, slice_method, spatial_size, nsp, int(image_size / seq_size))
            del gen_seq
        del seq
        g = model_generator(model=model.to(dtype), split_size=split_size, input_size=(mb, 3, image_size, image_size),
                            balance=balance, shape_list=shapes)
        g.ready_model(split_rank=comm.split_rank)
        gens.append(g)
    master = train_spatial_model_master(gens[0], gens[1], batch_size, spatial_size, num_spatial_parts, slice_method, comm1,
                                        comm2, LOCAL_DP_LP=1, parts=parts, ASYNC=True, replications=int(times / 2))
    sync = gems_comm.SyncAllreduce(comm1)
    n_img = batch_size * 2 * int(times / 2)

    def my_tile(x):
        if comm1.local_rank < P:
            return split_input(x, image_size, slice_method, comm1.local_rank, nsp)
        if comm2.local_rank < P:
            return split_input(x, image_size, slice_method, comm2.local_rank, nsp)
        return x

    perf = []
    for epoch in range(args.num_epochs):
        loss_sum = correct_sum = 0.0
        n = 0
        for inputs, labels in common.batches(args, image_size, n_img, args.steps):
            with common.StepTimer() as t:
                if args.enable_master_comm_opt:
                    loss, correct = master.run_step_allreduce(my_tile(inputs), labels, n % 2 == 1)
                    (master.train_model1 if n % 2 == 1 else master.train_model2).update()
                else:
                    loss, correct = master.run_step(my_tile(inputs), labels)
                    sync.apply_allreduce_master_master(gens[0], gens[1], comm1, comm2)
                    master.train_model1.update()
                    master.train_model2.update()
            loss_sum += loss
            correct_sum += correct
            n += 1
            if comm2.local_rank == 0:
                print("Epoch: %d images per sec:%s" % (epoch, n_img / t.seconds), flush=True)
                perf.append(n_img / t.seconds)
            if comm2.local_rank == comm1.size - 1:
                print("Step :%d, LOSS: %s, Global loss: %s Acc: %s" % (n - 1, loss, loss_sum / n, correct), flush=True)
        if comm2.local_rank == comm1.size - 1 and n:
            print("Epoch %d Global loss: %s Acc %s" % (epoch, loss_sum / n, correct_sum / n), flush=True)
    if comm2.local_rank == 0:
        common.report(perf)
    import torch.distributed as dist
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main(common.pop_model_flag(sys.argv, "resnet"))
