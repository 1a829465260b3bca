"""Data-parallel gradient exchange: one process per GPU, flat gradient buffers, bucketed
all-reduce launched from grad-ready hooks so that the exchange overlaps the rest of backward.

The reference is single-process (SURVEY.md §2.1); this is the one collective the sharded path
needs (§8e): average D's gradients after d_loss.backward() and G's after g_loss.backward().
Local BatchNorm statistics (= the reference run at the per-rank batch) and per-rank z/tau draws; with --sync-bn the
BatchNorm passes all-reduce their fp64 channel sums instead (ops.state.bn_group), so the statistics are those of the
global batch and every rank applies the same update to the running statistics.
torch.distributed does the plumbing (NCCL over NVLink on the GPUs; gloo in the CPU tests).
"""
import torch
import torch.distributed as dist


class BucketedAllReduce:
    """All-reduce (sum) of a flat gradient buffer in `num_buckets` contiguous slices.

    `params`/`offsets` describe where each parameter's gradient lives in `flat_grad`.  Backward
    produces gradients roughly in reverse registration order, so buckets are cut over the
    reversed list; a bucket's collective starts (async) when its last gradient has been
    accumulated.  The caller scales the loss by 1/world_size, so SUM yields the average.
    """

    def __init__(self, params, offsets, flat_grad, num_buckets=2, group=None):
        self.flat_grad, self.group = flat_grad, group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        order = sorted(range(len(params)), key=lambda i: offsets[i], reverse=True)
        total = flat_grad.numel()
        target = max(1, -(-total // max(1, num_buckets)))
        self.buckets, cur, lo, hi = [], [], None, None
        for i in order:
            n = params[i].numel()
            cur.append(i)
            lo = offsets[i] if lo is None else min(lo, offsets[i])
            hi = offsets[i] + n if hi is None else max(hi, offsets[i] + n)
            if hi - lo >= target:
                self.buckets.append((lo, hi, cur))
                cur, lo, hi = [], None, None
        if cur:
            self.buckets.append((lo, hi, cur))
        # widen slices so that together they cover the whole buffer (alignment padding included)
        self.buckets.sort(key=lambda b: b[0])
        fixed, start = [], 0
        for k, (lo, hi, members) in enumerate(self.buckets):
            end = total if k == len(self.buckets) - 1 else self.buckets[k + 1][0]
            fixed.append((start, end, members))
            start = end
        self.buckets = fixed
        self.bucket_of = {}
        for b, (_, _, members) in enumerate(self.buckets):
            for i in members:
                self.bucket_of[i] = b
        self.pending = [0] * len(self.buckets)
        self.works = []
        self.enabled = False
        self._hooks = [p.register_post_accumulate_grad_hook(self._make_hook(i)) for i, p in enumerate(params)]

    def _make_hook(self, i):
        def hook(_param):
            if not self.enabled or self.world == 1:
                return
            b = self.bucket_of[i]
            self.pending[b] -= 1
            if self.pending[b] == 0:
                lo, hi, _ = self.buckets[b]
                self._join()
                self.works.append(dist.all_reduce(self.flat_grad[lo:hi], group=self.group, async_op=True))
        return hook

    @staticmethod
    def _join():
        """The in-place weight-gradient kernels run on a side stream (ops._wgrad_direct): the collective, which is
        ordered after the launching stream only, must wait for them too."""
        if torch.cuda.is_available():
            from . import ops
            ops.join_all_streams(clear=False)

    def begin(self):
        """Arm the hooks for one backward pass."""
        self.enabled = True
        self.works = []
        self.pending = [len(m) for _, _, m in self.buckets]

    def finish(self):
        """Launch any bucket whose hooks did not all fire (unused parameters) and wait for all."""
        if self.world > 1:
            for b, left in enumerate(self.pending):
                if left > 0:
                    lo, hi, _ = self.buckets[b]
                    self._join()
                    self.works.append(dist.all_reduce(self.flat_grad[lo:hi], group=self.group, async_op=True))
                    self.pending[b] = 0
            for w in self.works:
                w.wait()
        self.works = []
        self.enabled = False

    def remove(self):
        for h in self._hooks:
            h.remove()


def shutdown(trainers=(), timeout_s=10.0):
    """Leave a data-parallel job without hanging: release the trainers' CUDA graphs (they hold captured NCCL kernels),
    then destroy the process group from a helper thread and give up on it after `timeout_s` (the caller is expected to
    exit the process next; a communicator that refuses to die must not keep a finished job alive)."""
    import threading
    for t in trainers:
        if hasattr(t, 'release_graphs'):
            t.release_graphs()
    if not (dist.is_available() and dist.is_initialized()):
        return True
    th = threading.Thread(target=dist.destroy_process_group, daemon=True)
    th.start()
    th.join(timeout_s)
    return not th.is_alive()


def shard_batch(global_batch, world, rank):
    """Contiguous per-rank slice of a global batch (strong-scaling helper)."""
    per = global_batch // world
    return slice(rank * per, (rank + 1) * per)
