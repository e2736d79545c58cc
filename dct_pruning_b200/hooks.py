"""Forward-hook side of the scoring path: every hook site of a net live at once.

Replaces the three hook functions and their module-global accumulators in
/root/reference/utils/common.py:

    get_feature_hook              :262-277   'O'  all channels of the module output
    get_feature_hook_densenet     :280-293   'D'  last 12 channels of the output
    get_feature_hook_u2net_input  :296-309   'I'  all channels of input[0]
    feature_result / total        :258-259   ->   one flat fp64 device accumulator per session

Each hook call is one asynchronous `dctp_score_accum(_ex)` launch on the current torch stream:
the activation is read once where cuDNN left it (NCHW fp32, or bf16 / fp16 under torch.autocast,
any batch/channel stride), no
coefficient tensor or per-slice value ever reaches host memory, and nothing synchronises
until `finalize()`.  The reference runs one forward sweep per site; registering all sites
together gives the same numbers on fixed inputs with one forward per batch.

There is no CPU path: a hook fired on a CPU tensor raises.
"""
import struct

import numpy as np
import torch

from . import _lib
from .sites import DENSENET_WINDOW, VARIANT_INPUT, VARIANT_LAST12, hook_sites, resolve_module


try:                                        # the raw handle of a device's current stream without building a torch.cuda.Stream object
    _raw_stream = torch._C._cuda_getCurrentRawStream
except AttributeError:                      # pragma: no cover - older / newer torch without the private accessor
    def _raw_stream(device_index):
        return torch.cuda.current_stream(device_index).cuda_stream

_SITE = struct.Struct('QQii')               # dctp_site of include/dctp.h: x, accum, B, c_count (24 bytes)


def ctypes_char_array(n_sites):
    import ctypes
    return ctypes.c_char * (_SITE.size * n_sites)


class ScoreSession:
    # One launch per hook costs twice.  The host needs ~12 us per hook (Python, ctypes, driver), which bounds the CIFAR nets and
    # U^2-Netp's small stages; and every launch of the warp-specialised kernels pays ~8-10 us of prologue, pipeline fill and drain
    # on the GPU (profiles/r02_launches_bench_resnet50.csv: 10 us + bytes / 3.6 TB/s), 15 % of ResNet-50's step.  Activations
    # smaller than DEFER_BYTES are therefore held (a reference keeps them alive, nothing is copied) and scored together with the
    # other sites of the same map size in ONE launch (dctp_score_accum_multi, up to 16 sites): ResNet-50's 49 hooks become 8
    # launches, ResNet-56's 55 become 6, U^2-Netp's 118 about 25.  One group is kept per map size (U^2-Net's stages alternate
    # sizes); a group is launched when it is full; everything that is held at the end of the forward pass (a hook on the net
    # itself), when HELD_BYTES are held, and on flush().  The price is memory: up to HELD_BYTES of activations stay allocated
    # until their launch (ResNet-50 at batch 256: 4.3 GB for the ten 56x56 sites).  defer_bytes=0 restores one launch per hook.
    DEFER_BYTES = 1 << 30
    MAX_PENDING = 16
    HELD_BYTES = 8 << 30

    def __init__(self, net, net_name, path='auto', capacity=1 << 18, sites=None, defer_bytes=None, op='dct2'):
        # op: the per-slice reduction - 'dct2' (common.py:267, the product), or one of the alternatives the reference keeps beside
        # it: 'rank' (:268, HRank), 'rank_sq' (:268 followed by the unchanged cnt_score), 'dct3' (:269, one value per site)
        if op not in _lib.OPS:
            raise ValueError('unknown scoring op %r (one of %s)' % (op, ', '.join(_lib.OPS)))
        self.op = op
        self.net = net
        self.net_name = net_name
        self.sites = list(hook_sites(net_name, net) if sites is None else sites)
        self.path = _lib.PATHS[path] if isinstance(path, str) else int(path)
        self.capacity = capacity
        self.flat = None                      # fp64 [capacity + 1]; last used slot (+1) carries the image count
        self.used = 0
        self.slots = [None] * len(self.sites)  # (offset, channels scored)
        self.images = [0] * len(self.sites)
        self.handles = []
        self.lib = _lib.load()
        self._score_accum = self.lib.dctp_score_accum
        self._score_accum_ex = self.lib.dctp_score_accum_ex     # 16-bit activations (dtype after the pointer)
        self._score_op = self.lib.dctp_score_op
        self._plans = [None] * len(self.sites)
        self._planned = False                 # plan_layout() ran: slots exist for every site, in site order
        self.defer_bytes = self.DEFER_BYTES if defer_bytes is None else int(defer_bytes)
        self._pending = {}                    # (H, W, device index, stream, dtype) -> [(tensor kept alive, address of its first scored map,
        self._held = 0                        #                                   B, c_count, accumulator address)]; bytes held
        self._score_multi = self.lib.dctp_score_accum_multi_ex
        self.launches = 0
        # The forward pass of the CIFAR nets is bound by the host (~20 us per module call), so what a hook costs the host is what it costs
        # end to end.  After a site's first firing everything that depends only on the activation's geometry is remembered here:
        # (shape, strides, device index, map bytes, byte offset of the first scored map, B, c_count, accumulator address, H, W, dtype)
        self._fast = [None] * len(self.sites)
        self._site_buf = bytearray(_SITE.size * self.MAX_PENDING)
        self._site_arr = (ctypes_char_array(self.MAX_PENDING)).from_buffer(self._site_buf)

    # ------------------------------------------------------------------ registration
    def register(self):
        if self.handles:
            raise RuntimeError('hooks already registered')
        from .dist import world_size
        if world_size() > 1 and not self._planned:
            # every rank runs this same line, so all of them fail here, before any forward pass and before the collective
            raise RuntimeError('multi-rank run: call plan_layout(example) before registering the hooks, so that every rank holds the '
                               'same accumulator layout even if its shard of the batches is empty (generate.score_session does)')
        for idx, site in enumerate(self.sites):
            module = resolve_module(self.net, site.module)
            self.handles.append(module.register_forward_hook(self._make_hook(idx, site)))
        # held activations are scored when the forward pass they belong to ends: nothing is kept across batches, so the caching
        # allocator sees the same allocation pattern every step
        self.handles.append(self.net.register_forward_hook(lambda module, inputs, output: self.flush()))
        return self

    def remove(self):
        self.flush()
        for h in self.handles:
            h.remove()
        self.handles = []

    def __enter__(self):
        return self.register()

    def __exit__(self, *exc):
        self.remove()

    def _make_hook(self, idx, site):
        take_input = site.variant == VARIANT_INPUT

        def hook(module, inputs, output):
            self.score(idx, inputs[0] if take_input else output)
        return hook

    # ------------------------------------------------------------------ one hook firing
    def score(self, idx, t):
        fast = self._fast[idx]
        if (fast is not None and t.shape == fast[0] and t.stride() == fast[1] and t.dtype is fast[10] and t.is_cuda
                and fast[3] < self.defer_bytes):
            first = t.data_ptr() + fast[4]
            if first % 16 == 0 and t.device.index == fast[2]:
                B = fast[5]
                key = (fast[8], fast[9], fast[2], _raw_stream(fast[2]), fast[11])
                group = self._pending.get(key)
                if group is None:
                    group = self._pending[key] = []
                group.append((t, first, B, fast[6], fast[7]))
                self._held += fast[3]
                if len(group) >= self.MAX_PENDING:
                    self.flush(key)
                elif self._held > self.HELD_BYTES:
                    self.flush()
                self.images[idx] += B
                return
        if not t.is_cuda:
            raise RuntimeError('dct_pruning_b200 scores on CUDA only (site %r fired on %s); there is no CPU fallback'
                               % (self.sites[idx].module, t.device))
        if t.dim() != 4:
            raise ValueError('site %r: expected an NCHW activation, got shape %s' % (self.sites[idx].module, tuple(t.shape)))
        dtype = _lib.dtype_code(t.dtype)
        if dtype is None or (dtype != _lib.DTYPE_F32 and self.op != 'dct2'):
            t = t.float()                     # the reference scores in fp32 (common.py:233,289); the DCT energy reads 16-bit maps itself
            dtype = _lib.DTYPE_F32
        sb, sc, sh, sw = t.stride()
        B, C, H, W = t.shape
        if sw != 1 or sh < W:
            t = t.contiguous()
            sb, sc, sh, sw = t.stride()
        plan = self._plans[idx]
        if plan is None or plan[0] != C:      # (channels, c_begin, c_count, accumulator address): fixed after the first firing
            if self.sites[idx].variant == VARIANT_LAST12:
                if C < DENSENET_WINDOW:
                    raise ValueError('site %r: DenseNet window needs >= %d channels, got %d'
                                     % (self.sites[idx].module, DENSENET_WINDOW, C))
                c_begin, c_count = C - DENSENET_WINDOW, DENSENET_WINDOW
            else:
                c_begin, c_count = 0, C
            off = self._slot(idx, 1 if self.op == 'dct3' else c_count, t.device)
            plan = self._plans[idx] = (C, c_begin, c_count, self.flat.data_ptr() + 8 * off)
        stream = _raw_stream(t.device.index)
        c_begin, c_count = plan[1], plan[2]
        if self.op != 'dct2':                 # the alternative ops: one launch per hook, same accumulator plumbing
            with torch.cuda.device(t.device):
                code = self._score_op(_lib.OPS[self.op], t.data_ptr(), B, H, W, sb, sc, sh, c_begin, c_count, plan[3], None, stream)
            if code:
                _lib.check(code)
            self.images[idx] += B
            self.launches += 1
            return
        dense = sh == W and sc == H * W and (B == 1 or (c_count == C and sb == C * H * W))
        es = t.element_size()
        if (self.defer_bytes and dense and H == W and self.path == _lib.PATH_AUTO and es * B * c_count * H * W < self.defer_bytes
                and (t.data_ptr() + es * c_begin * sc) % 16 == 0):
            key = (H, W, t.device.index, stream, dtype)
            group = self._pending.setdefault(key, [])
            group.append((t, t.data_ptr() + es * c_begin * sc, B, c_count, plan[3]))
            self._held += es * B * c_count * H * W
            self._fast[idx] = (t.shape, t.stride(), t.device.index, es * B * c_count * H * W, es * c_begin * sc, B, c_count, plan[3], H, W,
                               t.dtype, dtype)
            if len(group) >= self.MAX_PENDING:
                self.flush(key)
            elif self._held > self.HELD_BYTES:
                self.flush()
            self.images[idx] += B
            return
        # launch on the activation's own device and on that device's current stream (the hook may fire while another
        # device is current); the library refuses a device other than the one it was initialised on
        args = (B, H, W, sb, sc, sh, plan[1], plan[2], plan[3], None, None, self.path, stream)
        if t.device.index != torch.cuda.current_device():
            with torch.cuda.device(t.device):
                code = self._score_accum(t.data_ptr(), *args) if dtype == _lib.DTYPE_F32 else self._score_accum_ex(t.data_ptr(), dtype, *args)
        else:
            code = self._score_accum(t.data_ptr(), *args) if dtype == _lib.DTYPE_F32 else self._score_accum_ex(t.data_ptr(), dtype, *args)
        if code:
            _lib.check(code)
        self.images[idx] += B
        self.launches += 1

    def flush(self, key=None):
        """Score the held activations (one launch per 16 sites of a map size) and let go of them; `key`: one group only."""
        keys = [key] if key is not None else list(self._pending)
        for k in keys:
            pending = self._pending.pop(k, None)
            if not pending:
                continue
            H, W, dev_index, stream, dtype = k
            buf, off, map_bytes = self._site_buf, 0, (4 if dtype == _lib.DTYPE_F32 else 2) * H * W
            for _, x_ptr, B, c_count, acc_ptr in pending:             # dctp_site records packed in place (ctypes field stores are slow)
                _SITE.pack_into(buf, off, x_ptr, acc_ptr, B, c_count)
                off += _SITE.size
                self._held -= map_bytes * B * c_count
            sites = self._site_arr
            if dev_index != torch.cuda.current_device():
                with torch.cuda.device(dev_index):
                    code = self._score_multi(sites, len(pending), H, W, dtype, stream)
            else:
                code = self._score_multi(sites, len(pending), H, W, dtype, stream)
            if code:
                _lib.check(code)
            self.launches += 1

    def _slot(self, idx, c_count, device):
        if self.flat is None:
            if torch.device(device).type == 'cuda':
                with torch.cuda.device(device):
                    _lib.check(self.lib.dctp_init())
            self.flat = torch.zeros(self.capacity + 1, dtype=torch.float64, device=device)
        slot = self.slots[idx]
        if slot is None:
            if self.used + c_count > self.capacity:
                raise RuntimeError('score accumulator capacity %d exceeded' % self.capacity)
            slot = self.slots[idx] = (self.used, c_count)
            self.used += c_count
        elif slot[1] != c_count:
            raise ValueError('site %r changed width: %d -> %d channels' % (self.sites[idx].module, slot[1], c_count))
        return slot[0]

    def plan_layout(self, example):
        """Allocate every site's accumulator slot ahead of the run, in site order, from one shape-only forward pass of
        `example` (a [1,3,S,S] tensor on the net's device; nothing is scored).  Under torchrun every rank calls this, so all
        ranks hold the same flat layout and enter the run's single all-reduce even when a rank's shard of the batches is
        empty (batch size smaller than the world size)."""
        shapes = [None] * len(self.sites)
        taps = []
        for idx, site in enumerate(self.sites):
            def tap(module, inputs, output, idx=idx, take_input=(site.variant == VARIANT_INPUT)):
                shapes[idx] = tuple((inputs[0] if take_input else output).shape)
            taps.append(resolve_module(self.net, site.module).register_forward_hook(tap))
        live, self.handles = self.handles, []
        for h in live:
            h.remove()
        try:
            with torch.no_grad():
                self.net(example)
        finally:
            for h in taps:
                h.remove()
            if live:
                self.register()
        for idx, (site, shape) in enumerate(zip(self.sites, shapes)):
            if shape is None:
                continue
            C = shape[1]
            c_count = DENSENET_WINDOW if site.variant == VARIANT_LAST12 else C
            self._slot(idx, 1 if self.op == 'dct3' else c_count, example.device)
        self._planned = True
        return self

    # ------------------------------------------------------------------ CUDA-graph replay (launch-bound nets)
    def capture(self, example, warmup=2):
        """Capture one forward pass with every hook launch in a CUDA graph and return `replay(x)`.

        For the CIFAR-sized nets the scoring pass is launch-bound (tens of hooks over a few-millisecond
        forward); a graph removes the per-launch host cost of both the forward and the hooks.  `example`
        fixes shape and device; hooks must be registered (use inside `with session:`).  Each `replay(x)`
        scores one more batch, exactly like calling `net(x)` with the hooks live."""
        if not self.handles:
            raise RuntimeError('register the hooks before capturing (with session: ...)')
        if any(self.images):
            raise RuntimeError('capture() restarts the run (its warm-up passes are discarded with reset()); call it before the '
                               'first batch is scored, not after %d images' % max(self.images))
        static_in = example.detach().clone()
        side = torch.cuda.Stream(device=static_in.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(max(1, warmup)):             # allocates accumulator slots, uploads bases, warms cuDNN
                self.net(static_in)
            self.flush()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize(static_in.device)
        self.reset()
        before = list(self.images)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph), torch.no_grad():
            self.net(static_in)
            self.flush()                                # the held sites' launches belong to the graph
        per_replay = [after - b for after, b in zip(self.images, before)]
        self.images = before                            # the capture pass itself did not run
        self._graph = graph                             # keep alive

        def replay(x):
            static_in.copy_(x, non_blocking=True)
            graph.replay()
            for i, n in enumerate(per_replay):
                self.images[i] += n
        return replay

    def prepare(self, sides):
        """Upload the cosine bases for the given map sides ahead of time (keeps hooks capture-safe)."""
        for s in sides:
            h, w = (s, s) if isinstance(s, int) else s
            _lib.check(self.lib.dctp_prepare(h, w))

    def reset(self):
        """Start a new run (the reference's reset of feature_result/total, common.py:396-397)."""
        self._pending, self._held = {}, 0               # held sites belong to the run that is being discarded
        if self.flat is not None:
            self.flat.zero_()
        self.images = [0] * len(self.sites)

    # ------------------------------------------------------------------ end of run
    def finalize(self, group=None, check=True):
        """Sum over ranks (one all-reduce of the flat buffer), divide by the image count, cast to
        fp32.  Returns {file_stem: float32 numpy vector}, the payload of the reference's np.save calls."""
        device_scores = self.finalize_device(group=group, check=check)
        host = device_scores.cpu().numpy()
        return self.split_files(host)

    def reduce_sums(self, group=None):
        """The run's one collective: the flat fp64 sums, with the image count in the slot after the last score, summed over
        the ranks (a no-op in a single process).  Every rank enters it - also one whose shard was empty (its hooks never
        fired: zeros, count 0; `plan_layout` gave it the layout) - and the consistency checks run AFTER it, so that a bad
        rank cannot leave the others waiting in NCCL.  Returns the global image count."""
        from .dist import allreduce_sums, world_size
        self.flush()
        fired = sorted(set(n for n, s in zip(self.images, self.slots) if s is not None))
        n = self.used
        problem = None
        if self.flat is None:
            if world_size(group) > 1:
                problem = 'this rank holds no accumulator layout (call plan_layout() before a multi-rank run)'
            else:
                raise RuntimeError('no hook fired: nothing to finalize')
        elif len(fired) > 1:
            problem = 'hook sites saw different image counts: %s' % fired
        if self.flat is not None:
            self.flat[n] = float(fired[0]) if len(fired) == 1 else float('nan')
            allreduce_sums(self.flat[:n + 1], group=group)
        if problem is not None:
            raise RuntimeError(problem)
        n_images = float(self.flat[n].item())
        if not n_images > 0:                                   # nan (a rank reported a problem) or nothing scored anywhere
            raise RuntimeError('no hook fired on any rank (or a rank reported inconsistent image counts): nothing to finalize')
        self.n_images = n_images
        return n_images

    def finalize_device(self, group=None, check=True):
        n_images = self.reduce_sums(group=group)
        n = self.used
        out = torch.empty(n, dtype=torch.float32, device=self.flat.device)
        with torch.cuda.device(self.flat.device):
            _lib.check(self.lib.dctp_finalize(_lib.ptr(self.flat), n_images, _lib.ptr(out), n,
                                              torch.cuda.current_stream(self.flat.device).cuda_stream))
            if check:
                _lib.check(self.lib.dctp_check(torch.cuda.current_stream(self.flat.device).cuda_stream))
        return out

    def split_files(self, host_scores):
        files = {}
        for site, slot in zip(self.sites, self.slots):
            if slot is None:
                continue
            vec = host_scores[slot[0]:slot[0] + slot[1]]
            for f in site.files:
                whole = f.lo is None or self.op == 'dct3'        # dct3: one value per site, no per-branch slices
                files[f.stem] = np.array(vec if whole else vec[f.lo:f.hi], dtype=np.float32, copy=True)
        return files

    def file_segments(self):
        """[(file_stem, offset into the flat score vector, length)] in site order."""
        segs = []
        for site, slot in zip(self.sites, self.slots):
            if slot is None:
                continue
            for f in site.files:
                lo, hi = (0, slot[1]) if (f.lo is None or self.op == 'dct3') else (f.lo, f.hi)
                segs.append((f.stem, slot[0] + lo, hi - lo))
        return segs
