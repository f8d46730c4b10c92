"""The HiD-VAE training micro-step as CUDA graphs (train_hidvae.py:700-770 of the reference, one replay instead of the
several hundred kernel launches and Python dispatches of an eager step).

A step at the batch sizes HiD-VAE trains with (64 ... 8192 items) is launch-bound: the encoder / decoder / tag-head
layers, the fused quantiser kernels and their autograd nodes are ~1,000 launches of a few microseconds each, and the
GPU waits for Python between them.  `GraphedTrainStep` captures

    graph 1   batch gather (dataset[idx]) -> HRqVae.forward -> loss.backward() into the flat gradient buffer
              (+ the logged statistics as one 7-vector)
    graph 2   optimizer.step()            (AdamW with capturable=True and tensor learning rates)

once, after a few eager warm-up steps on the capture stream, and replays them.  Between the two graphs the data-parallel
exchange runs eagerly: one NCCL all-reduce of the flat buffer (`FlatGradAllReduce.all_reduce`); with one process the two
replays are back to back.  Requirements, checked at construction: no fp16 loss scaling (its inf check reads back to the
host), a model whose forward is free of host synchronisation (HRqVae is: the tag losses are masked fixed-shape means, the
uniqueness loss and p_unique_ids are kernels), fixed batch size.  Dropout and mixup draws advance inside the graph through
PyTorch's graph-safe Philox offsets, and so do the Gumbel-softmax levels: under capture `ops.gumbel_apply` draws each level's
noise seed on the device, so every replay draws new noise, and the forward and backward of one replay read the same seed.
`gumbel_t` is a host scalar and is frozen at capture; the trainer's temperature is the constant 0.2 of the reference, so
nothing is lost there, but a temperature schedule would need a new capture per value.  No autograd graph of an EARLIER eager
step may still be alive when this is built (e.g. a kept `out.loss`): its AccumulateGrad nodes are bound to the stream they
ran on, and the capture would have to synchronise with it.  The warm-up steps are REAL optimisation
steps (with the gradient exchange): a run with `warmup` = 3 has made three steps when the constructor returns."""
from typing import Callable, Optional

import torch
from torch import Tensor

STAT_NAMES = ("loss", "reconstruction", "rqvae", "tag_align", "tag_pred", "tag_acc", "p_unique")


def step_statistics(out) -> Tensor:
    """The seven logged quantities of one step as a device vector (train_hidvae.py:773-800)."""
    return torch.stack([out.loss.detach(), out.reconstruction_loss.mean(), out.rqvae_loss.mean(), out.tag_align_loss.mean(),
                        out.tag_pred_loss.mean(), out.tag_pred_accuracy.mean(), out.p_unique_ids.float()])


class GraphedTrainStep:
    def __init__(self, model: torch.nn.Module, optimizer: torch.optim.Optimizer, grads, fetch: Callable[[Tensor], object],
                 batch_size: int, n_items: int, gumbel_t: float = 0.2, loss_divisor: float = 1.0,
                 autocast_dtype: Optional[torch.dtype] = None, generator: Optional[torch.Generator] = None, warmup: int = 3):
        """`fetch(idx)` returns the batch of the item indices `idx` [batch_size] (e.g. `dataset.__getitem__`); `grads` is the
        FlatGradAllReduce whose views are the parameters' `.grad`s."""
        self.model, self.optimizer, self.grads = model, optimizer, grads
        self.batch_size, self.n_items, self.generator = int(batch_size), int(n_items), generator
        dev = grads.flat.device
        for group in optimizer.param_groups:
            if not group.get("capturable", False):
                raise ValueError("GraphedTrainStep: build the optimizer with capturable=True (and tensor learning rates if a "
                                 "scheduler changes them): a plain AdamW step reads its step counter on the host")
        self.idx = torch.zeros(self.batch_size, dtype=torch.int64, device=dev)
        self.stats = torch.zeros(len(STAT_NAMES), device=dev)
        self.emb_norms = torch.zeros(len(getattr(model, "layers", [])) or 1, device=dev)   # mean |emb_out| per level (logged)

        def micro_step():
            batch = fetch(self.idx)
            with torch.autocast("cuda", dtype=autocast_dtype or torch.bfloat16, enabled=autocast_dtype is not None):
                out = model(batch, gumbel_t=gumbel_t)
            grads.backward(out.loss / loss_divisor)   # (one multi-tensor add into the flat buffer, not an add_ per parameter)
            self.stats.copy_(step_statistics(out))
            self.emb_norms.copy_(out.embs_norm.mean(dim=0))

        # warm-up on a side stream (lazy initialisations, cuBLAS workspaces, autograd buffers), then capture
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(max(warmup, 1)):
                self._draw()
                grads.zero()
                micro_step()
                grads.all_reduce()      # (ranks must stay in step during the warm-up too)
                optimizer.step()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        grads.check_views()
        self.g_step, self.g_opt = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        grads.zero()
        with torch.cuda.graph(self.g_step):      # (capture records, it does not run: no index draw is consumed here)
            micro_step()
        with torch.cuda.graph(self.g_opt, pool=self.g_step.pool()):
            optimizer.step()
        grads.check_views()

    def _draw(self) -> None:
        """This step's item indices (every rank draws its own, train_hidvae.py:213,233) into the graph's static buffer."""
        torch.randint(0, self.n_items, (self.batch_size,), device=self.idx.device, generator=self.generator, out=self.idx)

    def micro_step(self) -> Tensor:
        """Gather + forward + backward of one freshly drawn batch (gradients ACCUMULATE in the flat buffer: call
        `grads.zero()` before the first micro-step of an optimisation step).  Returns the statistics vector (static)."""
        self._draw()
        self.g_step.replay()
        return self.stats

    def optimizer_step(self) -> None:
        self.g_opt.replay()

    def __call__(self) -> Tensor:
        """zero -> one micro-step -> all-reduce -> optimizer step."""
        self.grads.zero()
        stats = self.micro_step()
        self.grads.all_reduce()
        self.optimizer_step()
        return stats
