"""PyTorch criteria on CUDA tensors, end to end on the device (SURVEY.md section 8(f) rank 1).

The reference's example (bindings/python/examples/pytorch_loss.py:19-102) moves the emissions to
the CPU, builds one Graph per utterance inside gtn.parallel_for and copies the gradients back.
Here the [B, T, C] CUDA tensor goes straight into the C ABI (`gtnb_ctc_loss`, device pointers in,
device gradients out) on the tensor's own CUDA stream; only the B losses visit the host.
"""
import ctypes as C

import numpy as np
import torch

from . import capi

_ctx_cache = {}


def _ctx_for(device, stream):
    key = (device.index, stream)
    if key not in _ctx_cache:
        _ctx_cache[key] = capi.Ctx(device.index, stream)
    return _ctx_cache[key]


class CTCLossFunction(torch.autograd.Function):
    """loss_b = forwardScore(e_b) - forwardScore(intersect(ctcGraph(target_b), e_b))  (benchmarks/ctc.cpp:150-158).

    emissions: float32 CUDA tensor [B, T, C] (unnormalised scores are fine: the normaliser is part of the loss);
    targets: list of 1-D int sequences; returns the mean loss over the batch (reduction="mean") or the [B] vector.
    """

    @staticmethod
    def forward(ctx, emissions, targets, blank=0, reduction="mean"):
        assert emissions.is_cuda and emissions.dtype == torch.float32 and emissions.dim() == 3
        e = emissions.contiguous()
        B, T, Cn = e.shape
        stream = torch.cuda.current_stream(e.device).cuda_stream
        g = _ctx_for(e.device, stream)
        lens = np.asarray([len(t) for t in targets], np.int32)
        cat = np.ascontiguousarray(
            np.concatenate([np.asarray(t, np.int32) for t in targets]) if B else np.zeros(0, np.int32), np.int32)
        losses = np.zeros(B, np.float32)
        grad = torch.empty_like(e)
        g._check(capi.lib().gtnb_ctc_loss(
            g.h, B, T, Cn, e.data_ptr(), 1, None, cat.ctypes.data_as(capi._i32p),
            lens.ctypes.data_as(capi._i32p), int(blank), losses.ctypes.data_as(capi._f32p),
            grad.data_ptr(), 1))
        out = torch.from_numpy(losses).to(e.device)
        ctx.save_for_backward(grad)
        ctx.reduction = reduction
        ctx.B = B
        return out.mean() if reduction == "mean" else out

    @staticmethod
    def backward(ctx, grad_output):
        (grad,) = ctx.saved_tensors
        if ctx.reduction == "mean":
            scale = grad_output / ctx.B
            return grad * scale, None, None, None
        return grad * grad_output.view(-1, 1, 1), None, None, None


def ctc_loss(emissions, targets, blank=0, reduction="mean"):
    return CTCLossFunction.apply(emissions, targets, blank, reduction)


class ASGLossFunction(torch.autograd.Function):
    """loss_b = forwardScore(compose(e_b, transitions)) - forwardScore(compose(compose(fal_b, transitions), e_b))
    (examples/asg.cpp:59-81, test/criterion_test.cpp:244-305) with ONE learned transitions graph shared by the
    minibatch -- and by all ranks: with torch.distributed initialised, the transition gradient of the local shard
    is all-reduced (sum) over NCCL, the multi-GPU form of Graph::addGrad under grad_lock (graph.cpp:96-100).

    emissions: float32 CUDA tensor [B, T, C]; transitions: float32 tensor [C + C*C] (start weights, then the
    C x C matrix, row = destination label) on any device; targets: list of 1-D int sequences.
    """

    @staticmethod
    def forward(ctx, emissions, transitions, targets, reduction="mean", allreduce=True):
        assert emissions.is_cuda and emissions.dtype == torch.float32 and emissions.dim() == 3
        e = emissions.contiguous()
        B, T, Cn = e.shape
        assert transitions.numel() == Cn + Cn * Cn
        stream = torch.cuda.current_stream(e.device).cuda_stream
        g = _ctx_for(e.device, stream)
        tw = np.ascontiguousarray(transitions.detach().to("cpu", torch.float32).numpy())
        lens = np.asarray([len(t) for t in targets], np.int32)
        cat = np.ascontiguousarray(
            np.concatenate([np.asarray(t, np.int32) for t in targets]) if B else np.zeros(0, np.int32), np.int32)
        losses = np.zeros(B, np.float32)
        tgrad = np.zeros(Cn + Cn * Cn, np.float32)
        grad = torch.empty_like(e)
        g._check(capi.lib().gtnb_asg_loss(
            g.h, B, T, Cn, e.data_ptr(), 1, tw.ctypes.data_as(capi._f32p), cat.ctypes.data_as(capi._i32p),
            lens.ctypes.data_as(capi._i32p), losses.ctypes.data_as(capi._f32p), grad.data_ptr(), 1,
            tgrad.ctypes.data_as(capi._f32p)))
        tg = torch.from_numpy(tgrad).to(e.device)
        ctx.world = 1
        if allreduce and torch.distributed.is_available() and torch.distributed.is_initialized():
            torch.distributed.all_reduce(tg, op=torch.distributed.ReduceOp.SUM)
            ctx.world = torch.distributed.get_world_size()
        out = torch.from_numpy(losses).to(e.device)
        ctx.save_for_backward(grad, tg)
        ctx.reduction = reduction
        ctx.B = B
        ctx.tdev = transitions.device
        return out.mean() if reduction == "mean" else out

    @staticmethod
    def backward(ctx, grad_output):
        grad, tg = ctx.saved_tensors
        if ctx.reduction == "mean":
            # the mean over the GLOBAL batch when the transition gradient was summed over the ranks
            scale = grad_output / ctx.B
            return grad * scale, (tg * (scale / ctx.world)).to(ctx.tdev), None, None, None
        # reduction "none": the incoming gradient is per utterance; the transition gradient was already summed
        # over the batch inside the kernel, which is only the chain rule's answer for a uniform grad_output
        assert bool((grad_output == grad_output.flatten()[0]).all()), \
            "reduction='none' supports a uniform upstream gradient (sum / mean of the losses)"
        return grad * grad_output.view(-1, 1, 1), (tg * grad_output.flatten()[0]).to(ctx.tdev), None, None, None


def asg_loss(emissions, transitions, targets, reduction="mean", allreduce=True):
    return ASGLossFunction.apply(emissions, transitions, targets, reduction, allreduce)


@torch.no_grad()
def ctc_align(emissions, targets, input_lengths=None, blank=0, arc_sorted=True):
    """CTC forced alignment: the best path of intersect(ctcGraph(target_b), emissions_b) (gtnb_ctc_align).

    emissions: float32 CUDA tensor [B, T, C]; targets: list of 1-D int sequences; input_lengths: per-utterance
    frame counts (sequence or tensor), default T.  Returns (labels int32 [B, T], states int32 [B, T],
    scores float32 [B]) on the emissions' device: the path's label and CTC graph node per frame (-1 past
    input_lengths[b] or when no path exists) and its viterbiScore (-inf without a path).  Runs on the current
    stream; no autograd.
    """
    assert emissions.is_cuda and emissions.dtype == torch.float32 and emissions.dim() == 3
    e = emissions.detach().contiguous()
    B, T, Cn = e.shape
    stream = torch.cuda.current_stream(e.device).cuda_stream
    g = _ctx_for(e.device, stream)
    lens = np.asarray([len(t) for t in targets], np.int32)
    cat = np.ascontiguousarray(
        np.concatenate([np.asarray(t, np.int32) for t in targets]) if B else np.zeros(0, np.int32), np.int32)
    il = None
    if input_lengths is not None:
        if torch.is_tensor(input_lengths):
            input_lengths = input_lengths.detach().cpu().numpy()
        il = np.ascontiguousarray(input_lengths, np.int32)
        assert il.shape == (B,)
    labels = torch.empty((B, T), dtype=torch.int32, device=e.device)
    states = torch.empty((B, T), dtype=torch.int32, device=e.device)
    scores = np.zeros(max(B, 1), np.float32)
    g._check(capi.lib().gtnb_ctc_align(
        g.h, B, T, Cn, e.data_ptr(), 1, None if il is None else il.ctypes.data_as(capi._i32p),
        cat.ctypes.data_as(capi._i32p), lens.ctypes.data_as(capi._i32p), int(blank), int(arc_sorted),
        labels.data_ptr(), states.data_ptr(), 1, scores.ctypes.data_as(capi._f32p)))
    return labels, states, torch.from_numpy(scores[:B]).to(e.device)
