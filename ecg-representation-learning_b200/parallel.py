"""
Data-parallel gradient exchange: one process per GPU, full replicas, batch sharded across ranks.

The reference is single-process / single-device (SURVEY.md 2.1), so this is new: the only exchange step of the
path is a SUM all-reduce of the flat fp32 gradient buffer.  Backward produces gradients top layer first, and the
flat buffer is laid out in forward order, so a bucket is a contiguous slice [offset(layer lo) : offset(layer hi+1))
that becomes final the moment layer `lo` finishes its backward.  Each bucket's NCCL all-reduce is issued
asynchronously (it runs on c10d's internal NCCL stream, ordered after the producing kernels through an event)
while the compute stream keeps running the backward of the layers below; the 1/world average is folded into the
clip + AdamW kernels (`hyper[8]`), so no extra pass touches the gradients.
"""
import torch
import torch.distributed as dist


def bucket_slices(layer_offsets, total, depth, bucket_layers, lowest=-1, span_lo=0):
    """[(trigger_layer, lo, hi)] in the order backward completes them.

    layer_offsets[l] = first element of layer l's parameters in the flat buffer (forward order); everything before
    layer 0 (pos, cls, patch embedding) belongs to trigger -1, everything after the last layer (head) to the first
    bucket.  (lowest, span_lo): the trainable span (`EcgVit.trainable_span`); the buckets cover [span_lo, total) and
    every trigger is a position that backward visits, the head's backward (trigger `depth`) when no encoder or
    embedding parameter is trainable."""
    out = []
    hi = total
    l = depth
    bottom = max(lowest, 0)
    while l > bottom:
        lo_layer = max(bottom, l - bucket_layers)
        lo = max(span_lo, layer_offsets[lo_layer])
        out.append((lo_layer, lo, hi))
        hi = lo
        l = lo_layer
    if lowest in (-1, depth):   # the embedding's bucket, or the head's alone
        out.append((lowest, span_lo, hi))
    return [(t, lo, hi) for (t, lo, hi) in out if hi > lo]


class BucketedGradReducer:
    def __init__(self, model=None, group=None, bucket_layers=1, flat_g=None, layer_offsets=None, depth=None, bf16=False):
        """bf16=True: every bucket is cast to bf16 (a contiguous slice of `flat_g16`) right before its all-reduce and the
        optimizer kernels read the reduced bf16 image; the fp32 buffer keeps receiving the split-K partial sums."""
        self.group = group
        span = None
        if model is not None:
            flat_g = model._flat_g
            depth = model.config.num_hidden_layers
            layer_offsets = [model._layout[f'l{l}.ln1.w'][0] for l in range(depth)]
            model._after_layer_backward = self.on_layer_done
            span = model.trainable_span()
        self.span_key = None if span is None else span.key
        self.flat_g = flat_g
        self.flat_g16 = torch.empty(flat_g.numel(), device=flat_g.device, dtype=torch.bfloat16) if bf16 else None
        if span is None:
            self.slices = bucket_slices(layer_offsets, flat_g.numel(), depth, bucket_layers)
        else:
            # buckets over the trainable span; a bucket that holds no trainable tensor is not exchanged
            self.slices = bucket_slices(layer_offsets, flat_g.numel(), depth, bucket_layers, span.lowest, span.lo)
            live = [o for k, (o, _, _, _) in model._layout.items() if k not in span.frozen]
            self.slices = [(t, lo, hi) for (t, lo, hi) in self.slices if any(lo <= o < hi for o in live)]
        self.by_trigger = {t: (lo, hi) for (t, lo, hi) in self.slices}
        self.works = []

    def begin(self):
        self.works = []

    def on_layer_done(self, layer):
        s = self.by_trigger.get(layer)
        if s is None:
            return
        lo, hi = s
        buf = self.flat_g[lo:hi]
        if self.flat_g16 is not None:
            if buf.is_cuda:
                from . import _lib
                _lib.check(_lib.load().ecgvit_cast_f32_to_bf16(buf.data_ptr(), self.flat_g16[lo:hi].data_ptr(), hi - lo,
                                                               torch.cuda.current_stream().cuda_stream), 'cast')
            else:
                self.flat_g16[lo:hi].copy_(buf)   # host-side tests of the bucketing logic (gloo)
            buf = self.flat_g16[lo:hi]
        self.works.append(dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=self.group, async_op=True))

    def finish(self):
        for w in self.works:
            w.wait()  # makes the current stream wait for the NCCL stream (no host block on CUDA)
        self.works = []
