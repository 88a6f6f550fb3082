#!/usr/bin/env python3
"""Flagship benchmark: MoE-layer training step (fwd + bwd + SGD) throughput, whole job, device-timed.

Config (BASELINE.json #2, weak scaling): helloworld model, top-2, 8 global experts (8/N per GPU), bf16,
model_dim 4096, hidden 14336, 16 x 512 = 8192 tokens per GPU, capacity_factor 1.0, synthetic data, random init.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29500 \
        bench.py --gpus 8 --steps 20 --warmup 5
    python bench.py --gpus 1 --steps 20 --warmup 5 --dump-outputs /tmp/out   # + the last step's results as .npy files
    python bench.py --impl reference ...      # the UNMODIFIED reference from baseline/_ref, same metric / config

Prints one JSON line on rank 0.
"""
import argparse
import gc
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))

MODEL_DIM, HIDDEN, GLOBAL_EXPERTS, TOP_K = 4096, 14336, 8, 2
BATCH, TOKENS = 16, 512


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', type=str, default='ours', choices=['ours', 'reference'])
    ap.add_argument('--model_dim', type=int, default=MODEL_DIM)
    ap.add_argument('--hidden', type=int, default=HIDDEN)
    ap.add_argument('--experts', type=int, default=GLOBAL_EXPERTS)
    ap.add_argument('--top', type=int, default=TOP_K)
    ap.add_argument('--overlap', type=int, default=1)
    ap.add_argument('--no_e2e', action='store_true')
    ap.add_argument('--expert_type', type=str, default='ffn')     # llama_ffn: Mixtral-style SwiGLU block (BASELINE config #3)
    ap.add_argument('--fp8', action='store_true')                  # ours only: e4m3 forward + data-gradient GEMMs
    ap.add_argument('--graph', default='auto', choices=['auto', 'off'])     # ours, 1 GPU: replay the whole step as one CUDA graph
    ap.add_argument('--fp8_mode', default='row', choices=['row', 'mx'])   # row scales (fused engine) or MX 32-element block scales
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last step computed (loss, input gradient, parameter '
                         'gradients and updated parameters) as DIR/<name>.npy, for output-for-output comparison of builds')
    return ap.parse_args()


DUMP_SAMPLE = 1 << 18      # elements kept of a larger array: every dump stays far below 64 MB


def dump_outputs(out_dir, loss, x, model):
    """Write the loss, the input gradient and every parameter's gradient and updated value as float32 (float64 for
    float64 tensors) .npy files.  An array of more than DUMP_SAMPLE elements is stored as a 1-D sample at fixed, seeded
    flat indices (the same for every run of the same shapes)."""
    import numpy as np
    import torch
    arrays = [('loss', loss), ('input_grad', x.grad)]
    for name, p in model.named_parameters():
        arrays += [('param.' + name, p), ('grad.' + name, p.grad)]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays:
        if t is None:
            continue
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randint(0, t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        t = t.to(torch.float64 if t.dtype == torch.float64 else torch.float32).cpu()
        np.save(os.path.join(out_dir, name + '.npy'), t.numpy())


def main():
    args = parse()
    if args.impl == 'reference':
        ref = os.path.join(ROOT, 'baseline', '_ref')
        if not os.path.isdir(os.path.join(ref, 'tutel')):
            print(json.dumps({'impl': 'reference', 'unavailable': 'baseline/_ref is not installed (pip install --target baseline/_ref /root/reference)'}))
            return
        sys.path.insert(0, ref)
        try:
            from tutel import moe as moe_api, net as net_api, system as system_api  # noqa
        except Exception as ex:  # noqa
            print(json.dumps({'impl': 'reference', 'unavailable': 'import failed: %r' % (ex,)}))
            return
    else:
        sys.path.insert(0, ROOT)
        from tutel_b200 import moe as moe_api, net as net_api, system as system_api  # noqa

    import torch
    import torch.distributed as dist
    import torch.nn.functional as F

    world = int(os.environ.get('WORLD_SIZE', '1'))
    assert world == args.gpus or world == 1 and args.gpus == 1, 'launch with torchrun --nproc-per-node %d' % args.gpus
    env = system_api.init_data_model_parallel(backend='nccl')
    rank, device = env.global_rank, env.local_device
    torch.cuda.set_device(device)
    torch.set_default_dtype(torch.bfloat16)

    assert args.experts % world == 0, 'global experts must divide over the GPUs'
    local_experts = args.experts // world

    class Model(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self._moe_layer = moe_api.moe_layer(
                gate_type={'type': 'top', 'k': args.top, 'fp32_gate': False, 'capacity_factor': 1.0},
                experts=dict({'type': args.expert_type, 'num_experts_per_device': local_experts,
                              'hidden_size_per_expert': args.hidden},
                             **({'activation_fn': (lambda x: F.relu(x))} if args.expert_type == 'ffn' else {}),
                             **({'fp8': args.fp8_mode} if (args.fp8 and args.impl == 'ours') else {})),
                model_dim=args.model_dim,
                scan_expert_func=lambda name, param: setattr(param, 'skip_allreduce', True),
                seeds=(1, rank + 1, 1),
                a2a_ffn_overlap_degree=args.overlap,
            )

        def forward(self, x):
            return F.log_softmax(torch.sum(self._moe_layer(x), dim=2), dim=1)

    model = Model().to(device)
    optimizer = torch.optim.SGD(model.parameters(), lr=1e-5)
    shared = [p for p in model.parameters() if not hasattr(p, 'skip_allreduce') and p.requires_grad]

    torch.manual_seed(rank)
    x_host = torch.randn([BATCH, TOKENS, args.model_dim], dtype=torch.float32).to(torch.bfloat16).pin_memory()
    y_host = torch.zeros(BATCH, dtype=torch.int64).pin_memory()
    # The layer's input requires a gradient (in a real network the MoE block is never the first layer): the step then
    # contains all six expert GEMMs - fwd 2, dgrad 2, wgrad 2 - and the input-gradient combine, in BOTH arms.
    x_dev, y_dev = x_host.to(device).requires_grad_(True), y_host.to(device)

    def step(x, y):
        optimizer.zero_grad()
        x.grad = None
        loss = F.nll_loss(model(x), y)
        loss.backward()
        if world > 1:
            for p in shared:
                p.grad /= world
                p.grad = net_api.simple_all_reduce(p.grad)
        optimizer.step()
        return loss

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxreduce(v):
        t = torch.tensor([v], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    launches0 = 0
    if args.impl == 'ours':
        from tutel_b200.ops import backend
    # ---------------- kernel-side number: inputs resident on the device ----------------
    sampler = None
    if rank == 0:
        try:
            # plain nvidia-smi poller (no kernels, no native code); loaded by file path so that the reference arm's process
            # never imports the tutel_b200 package
            import importlib.util
            spec = importlib.util.spec_from_file_location('_bench_timers', os.path.join(ROOT, 'tutel_b200', 'utils', 'timers.py'))
            timers = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(timers)
            sampler = timers.ClockSampler(device.index or 0).start()  # started early: nvidia-smi needs a moment to spin up
        except Exception:  # noqa
            sampler = None
    eager_step = step
    first_loss = float(step(x_dev, y_dev).item())          # loss of the very first step (same seeds in both arms)
    warm_done = 1
    for _ in range(max(args.warmup, 3) - 1):
        step(x_dev, y_dev)
        warm_done += 1
    sync()
    # ours, one GPU: nothing in a step touches the host, so the whole step (zero_grad, forward, loss, backward, SGD) is
    # recorded once with the framework's public `GraphedTrainStep` and replayed as ONE graph launch per step - the same
    # kernels do the same work, only the ~40 launches per step are issued by the GPU front end instead of Python.
    # (Multi-GPU steps number their peer-to-peer transactions on the host and are not captured; the reference's step
    # reads the capacity back to the host in every forward and cannot be captured at all.)
    graph_info = {'cuda_graph': False}
    if args.impl == 'ours' and world == 1 and args.graph == 'auto':
        try:
            from tutel_b200.utils.graph import GraphedTrainStep
            gstep = GraphedTrainStep(eager_step, x_dev, y_dev, warmup=2)
            warm_done += 3
            probe = float(gstep(x_dev, y_dev).item())
            assert probe == probe, 'graph replay produced a NaN loss'
            warm_done += 1

            def step(x, y):                       # noqa: F811 - same signature, replays the captured step
                return gstep(x, y)
            x_dev, y_dev = gstep.static_inputs    # resident inputs of the device-timed loop: no copy in front of a replay
            graph_info = {'cuda_graph': True, 'launches_per_graph_replay': gstep.launches_per_replay}
        except Exception as ex:  # noqa - capture not possible on this build: measure the eager step
            step = eager_step
            graph_info = {'cuda_graph': False, 'graph_capture_error': repr(ex)[:200]}
            torch.cuda.synchronize()
    # Keep warming (untimed) until the step time has converged: blocks of 4 steps, stop when two consecutive blocks agree
    # within 2 % on every rank (clocks, the power-cap controller and the allocator settle within a few dozen steps).
    # With --dump-outputs all 12 blocks run: every SGD step moves the weights, so the dumped step must be the same step
    # of the training run each time.
    prev_blk, warm_trace = None, []
    for _ in range(12):
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record()
        for _ in range(4):
            step(x_dev, y_dev)
        w1.record()
        sync()
        warm_done += 4
        blk = maxreduce(w0.elapsed_time(w1) / 4)
        warm_trace.append(round(blk, 3))
        if args.dump_outputs is None and prev_blk is not None and abs(blk - prev_blk) <= 0.02 * prev_blk:
            break
        prev_blk = blk
    if args.impl == 'ours':
        launches0 = backend.launch_count()
    # (both arms) no cyclic-garbage collection inside a timed region: with tightly coupled ranks one collector pause on any
    # rank stalls every rank
    gc.collect()
    gc.disable()
    t_wall0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step(x_dev, y_dev)
    e1.record()
    sync()
    t_wall1 = time.time()
    gc.enable()
    last_loss, last_x = loss, x_dev
    ms = maxreduce(e0.elapsed_time(e1))
    launches = (backend.launch_count() - launches0) if args.impl == 'ours' else None
    clocks = None
    if sampler is not None:
        sampler.stop()
        clocks = sampler.summary(t_wall0, t_wall1)

    # ---------------- end-to-end number: H2D of the step's inputs from pinned memory + D2H of the loss ----------------
    e2e = None
    if not args.no_e2e:
        # Every step's inputs are copied from pinned host memory (64 MiB + labels) and every step's loss is read back.
        # The copy for step i+1 is issued on a copy stream before step i is launched (double-buffered input
        # prefetch, plain torch in both arms), so it overlaps with compute; all `steps` copies are inside the region.
        copy_stream = torch.cuda.Stream()
        slots = [(torch.empty_like(x_dev).requires_grad_(True), torch.empty_like(y_dev)) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]

        def prefetch(i):
            xb, yb = slots[i % 2]
            with torch.cuda.stream(copy_stream), torch.no_grad():
                copy_stream.wait_event(done[i % 2])       # the step that last read this slot has finished
                xb.copy_(x_host, non_blocking=True)
                yb.copy_(y_host, non_blocking=True)
                ready[i % 2].record(copy_stream)

        # The loss of every step is copied to pinned host memory right behind the step (asynchronously) and consumed by
        # the host one step later - the way a training loop logs its loss without stalling the launch queue; every
        # step's result is read inside the timed region, the last one before the closing event.
        loss_host = [torch.empty((), dtype=torch.get_default_dtype()).pin_memory() for _ in range(2)]
        loss_ready = [torch.cuda.Event() for _ in range(2)]

        def run(n):
            last, pending = None, None
            prefetch(0)
            for i in range(n):
                if i + 1 < n:
                    prefetch(i + 1)
                torch.cuda.current_stream().wait_event(ready[i % 2])
                loss_i = step(*slots[i % 2])
                done[i % 2].record()
                with torch.no_grad():
                    loss_host[i % 2].copy_(loss_i.detach(), non_blocking=True)   # device -> host read of the step's result
                loss_ready[i % 2].record()
                if pending is not None:
                    loss_ready[pending].synchronize()
                    last = float(loss_host[pending])
                pending = i % 2
            loss_ready[pending].synchronize()
            last = float(loss_host[pending])
            return last

        for ev in done:
            ev.record()
        run(3)
        sync()
        gc.collect()
        gc.disable()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        last = run(args.steps)
        f1.record()
        sync()
        gc.enable()
        ms_e2e = maxreduce(f0.elapsed_time(f1))
        # the last step's loss as the host received it; a graph replay computes the gradient of its static input x_dev
        last_loss = loss_host[(args.steps - 1) % 2]
        last_x = x_dev if graph_info['cuda_graph'] else slots[(args.steps - 1) % 2][0]
        e2e = {'value': world * BATCH * TOKENS * args.steps / (ms_e2e * 1e-3), 'unit': 'tokens/s',
               'h2d_bytes_per_step': x_host.numel() * x_host.element_size() + y_host.numel() * y_host.element_size(),
               'd2h_bytes_per_step': loss_host[0].numel() * loss_host[0].element_size(), 'ms_per_step': ms_e2e / args.steps, 'last_loss': last,
               'loss_read': 'asynchronous D2H copy into pinned memory behind every step, consumed by the host one step later (same in both arms)',
               'input_pipeline': 'double-buffered H2D prefetch on a copy stream (same in both arms)'}

    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, last_loss, last_x, model)

    tokens = world * BATCH * TOKENS * args.steps
    value = tokens / (ms * 1e-3)
    mats = 3 if args.expert_type == 'llama_ffn' else 2
    # per GPU per step: `mats` expert GEMMs forward, 2 x `mats` backward (data + weight gradients; x.requires_grad)
    flops = 2.0 * mats * 3 * BATCH * TOKENS * args.model_dim * args.hidden * min(args.top, args.experts)
    out = {
        'metric': 'moe_layer_fwd_bwd_tokens_per_sec', 'value': value, 'unit': 'tokens/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': warm_done, 'warmup_requested': args.warmup, 'warmup_ms_per_step_trace': warm_trace, 'ms_per_step': ms / args.steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16' if not (args.fp8 and args.impl == 'ours') else 'bf16 (fp8 e4m3 expert GEMMs, %s scales)' % args.fp8_mode, 'data': 'synthetic (random tokens, random-init weights)',
        'impl': args.impl,
        'config': {'model': 'helloworld moe_layer top-%d %d-expert %s%s model_dim=%d hidden=%d' % (
            args.top, args.experts, 'ffn(relu)' if args.expert_type == 'ffn' else args.expert_type, (' fp8-' + args.fp8_mode) if args.fp8 else '', args.model_dim, args.hidden),
                   'global_batch': world * BATCH, 'seq_len': TOKENS, 'tokens_per_gpu': BATCH * TOKENS,
                   'parallelism': 'ep%d (%d local experts/GPU)' % (world, local_experts), 'capacity_factor': 1.0,
                   'step': 'zero_grad + fwd + nll_loss + bwd (incl. input gradient) + gate-grad all-reduce + SGD',
                   'l2': 'working set (weights %.1f GB + activations) exceeds the 126 MB L2; no explicit flush' % (
                       local_experts * 2 * args.model_dim * args.hidden * 2 / 1e9),
                   'a2a_ffn_overlap_degree': args.overlap, **graph_info},
        'tflops_per_gpu': flops / (ms / args.steps * 1e-3) * 1e-12,
        'clocks': clocks, 'e2e': e2e, 'gpu_launches': launches, 'loss': float(loss.item()), 'first_step_loss': first_loss,
    }
    if rank == 0:
        print(json.dumps(out))
    sys.stdout.flush()


if __name__ == '__main__':
    main()
