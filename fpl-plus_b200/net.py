"""Drop-in ``UNet2D5_dsbn`` for PyMIC's ``net_dict`` (reference:
PyMIC/pymic/net/net3d/unet2d5_dsbn.py:239-309, net_run_dsbn/dsbn.py:35-64).

Same constructor (``params`` dict), same ``forward(x, domain_label)``, same 484-entry
``state_dict`` (the torch ``nn`` modules below are used purely as parameter containers, created
in the reference's order so default initialisation under a given seed is identical), same
``nn.Dropout`` children for the agent's test-time-dropout hook (agent_seg.py:845-852).

The arithmetic is NOT torch: ``forward`` runs the whole network as one autograd node whose
forward/backward are sequences of sm_100a kernels behind the C ABI (tcgen05 implicit-GEMM convs,
fused DSBN+PReLU+dropout+pool kernels, skip/up tensors written straight into shared concat
buffers).  Activations live in bf16 C8-planar layout; images/logits stay NCDHW fp32.
"""
import ctypes
import os

import torch
import torch.nn as nn

from . import ops
from .ops import C8, call, ptr, stream_ptr


# ------------------------------------------------------------------------------------------
# parameter containers (state_dict compatible with the reference)
# ------------------------------------------------------------------------------------------
class DomainSpecificBatchNorm2d(nn.Module):
    def __init__(self, num_features, num_domains):
        super().__init__()
        self.bns = nn.ModuleList([nn.BatchNorm2d(num_features) for _ in range(num_domains)])


class DomainSpecificBatchNorm3d(nn.Module):
    def __init__(self, num_features, num_domains):
        super().__init__()
        self.bns = nn.ModuleList([nn.BatchNorm3d(num_features) for _ in range(num_domains)])


class ConvBlockND(nn.Module):
    """conv -> DSBN -> PReLU -> Dropout -> conv -> DSBN -> PReLU (unet2d5_dsbn.py:48-83)."""

    def __init__(self, in_channels, out_channels, num_domains=None, dim=2, dropout_p=0.5):
        super().__init__()
        self.conv2d_1 = nn.Conv2d(in_channels, out_channels, kernel_size=3, padding=1)
        self.conv2d_2 = nn.Conv2d(out_channels, out_channels, kernel_size=3, padding=1)
        self.conv3d_1 = nn.Conv3d(in_channels, out_channels, kernel_size=3, padding=1)
        self.conv3d_2 = nn.Conv3d(out_channels, out_channels, kernel_size=3, padding=1)
        self.bn2d1 = DomainSpecificBatchNorm2d(out_channels, num_domains)
        self.bn2d2 = DomainSpecificBatchNorm2d(out_channels, num_domains)
        self.bn3d1 = DomainSpecificBatchNorm3d(out_channels, num_domains)
        self.bn3d2 = DomainSpecificBatchNorm3d(out_channels, num_domains)
        self.dropout_p = dropout_p
        self.dropout = nn.Dropout(dropout_p)
        self.relu_1 = nn.PReLU()
        self.relu_2 = nn.PReLU()
        self.dim = dim
        self.in_channels, self.out_channels = in_channels, out_channels

    def units(self):
        """(conv, dsbn, prelu, dropout-or-None) for the two conv units in use."""
        if self.dim == 2:
            return ((self.conv2d_1, self.bn2d1, self.relu_1, self.dropout),
                    (self.conv2d_2, self.bn2d2, self.relu_2, None))
        return ((self.conv3d_1, self.bn3d1, self.relu_1, self.dropout),
                (self.conv3d_2, self.bn3d2, self.relu_2, None))


class DownBlock(nn.Module):
    def __init__(self, in_channels, out_channels, num_domains=None, dim=2, dropout_p=0.0, downsample=True):
        super().__init__()
        self.downsample, self.dim = downsample, dim
        self.conv = ConvBlockND(in_channels, out_channels, num_domains, dim, dropout_p)


class UpBlock(nn.Module):
    def __init__(self, in_channels1, in_channels2, out_channels, num_domains=None, dim=2, dropout_p=0.0,
                 bilinear=True):
        super().__init__()
        self.bilinear, self.dim = bilinear, dim
        self.conv2d = nn.Conv2d(in_channels1, in_channels2, kernel_size=1)
        self.conv3d = nn.Conv3d(in_channels1, in_channels2, kernel_size=1)
        self.trans2d = nn.ConvTranspose2d(in_channels1, in_channels2, kernel_size=2, stride=2)
        self.trans3d = nn.ConvTranspose3d(in_channels1, in_channels2, kernel_size=2, stride=2)
        self.conv = ConvBlockND(in_channels2 * 2, out_channels, num_domains, dim, dropout_p)


# ------------------------------------------------------------------------------------------
# execution engine
# ------------------------------------------------------------------------------------------
class _Unit(object):
    """One conv + DSBN + PReLU (+dropout) stage and where its tensors live."""

    def __init__(self, name, conv, dsbn, prelu, dropout, kd, is_stem=False):
        self.name, self.conv, self.dsbn, self.prelu, self.dropout = name, conv, dsbn, prelu, dropout
        self.kd, self.is_stem = kd, is_stem
        self.cin, self.cout = conv.in_channels, conv.out_channels


class _Workspace(object):
    def __init__(self, device):
        self.device = device
        self.t = {}

    def get(self, name, shape, dtype):
        t = self.t.get(name)
        if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype:
            t = torch.empty(shape, dtype=dtype, device=self.device)
            self.t[name] = t
        return t

    def c8(self, name, n, d, c, h, w):
        return self.get(name, (n, d, c // 8, h, w, 8), torch.bfloat16)


class _Lease(object):
    """Returns a workspace to the pool when the autograd node that used it is freed."""

    def __init__(self, pool, ws):
        self.pool, self.ws = pool, ws

    def __del__(self):
        try:
            self.pool.append(self.ws)
        except Exception:
            pass


class _Plan(object):
    """The kernel of every launch site of one pass (UNet2D5_dsbn._plan) and the weight images they read."""

    def __init__(self):
        self.fwd, self.dgrad, self.wgrad = {}, {}, {}   # conv unit name -> kernel
        self.head = None                                # "cc" (csrc/head.cu), "tc" (zero-padded), "direct"
        self.up = []                                    # up1..up4: "proj" (bilinear), "tc" / "direct" (transposed conv)
        self.images = []                                # (kind, conv, transpose or convT mode, kd): prepare() stages them
        self.eval_fuse = False                          # conv + eval-mode BatchNorm + PReLU in one kernel (EpiAct)


class UNet2D5_dsbn(nn.Module):
    """DSBN 2.5D/3D U-Net; see module docstring.  ``params`` keys: in_chns, feature_chns[5],
    dropout[5], conv_dims[5] (2 or 3), class_num, bilinear, num_domains (extra keys ignored)."""

    def __init__(self, params):
        super().__init__()
        self.params = params
        self.in_chns = params['in_chns']
        self.ft_chns = list(params['feature_chns'])
        self.dropout = list(params['dropout'])
        self.dims = list(params['conv_dims'])
        self.n_class = params['class_num']
        self.bilinear = params['bilinear']
        self.num_domains = params['num_domains']
        assert len(self.ft_chns) == 5
        ft, nd, dm, dp = self.ft_chns, self.num_domains, self.dims, self.dropout
        self.block0 = DownBlock(self.in_chns, ft[0], nd, dm[0], dp[0], True)
        self.block1 = DownBlock(ft[0], ft[1], nd, dm[1], dp[1], True)
        self.block2 = DownBlock(ft[1], ft[2], nd, dm[2], dp[2], True)
        self.block3 = DownBlock(ft[2], ft[3], nd, dm[3], dp[3], True)
        self.block4 = DownBlock(ft[3], ft[4], nd, dm[4], dp[4], False)
        self.up1 = UpBlock(ft[4], ft[3], ft[3], nd, dm[3], dropout_p=dp[3], bilinear=self.bilinear)
        self.up2 = UpBlock(ft[3], ft[2], ft[2], nd, dm[2], dropout_p=dp[2], bilinear=self.bilinear)
        self.up3 = UpBlock(ft[2], ft[1], ft[1], nd, dm[1], dropout_p=dp[1], bilinear=self.bilinear)
        self.up4 = UpBlock(ft[1], ft[0], ft[0], nd, dm[0], dropout_p=dp[0], bilinear=self.bilinear)
        self.out_conv = nn.Conv3d(ft[0], self.n_class, kernel_size=(1, 3, 3), padding=(0, 1, 1))
        # engine state (not part of state_dict)
        self._pool = []
        self._infer_ws = None
        self._img_cache = {}
        self._dropout_masks = None      # {unit name: uint8 keep mask, dense C8-planar order} (parity tests)
        self._rng_dev = None            # int64[1] device seed read by the dropout kernels inside CUDA graphs
        self._rng_lanes = {}
        self._cur_lane = 0
        self._seed_from_device = False
        self._graphs = {}               # (shape, domain, mode) -> _GraphedForward (no-grad forwards)
        self._graph_ws_keep = []        # workspaces baked into captured graphs: never recycled
        self._infer_wss = {}            # eager no-grad workspaces per graph lane
        self.cuda_graphs = os.environ.get("FPL_CUDA_GRAPH", "1") != "0"
        # the reference paths tests compare against: "direct" = CUDA-core convolutions, the two-kernel inference
        # epilogue, gradients handed back to autograd
        self.conv_impl = os.environ.get("FPL_CONV_IMPL", "tc")
        self.eval_fuse = os.environ.get("FPL_EVAL_FUSE", "1") != "0"
        self.grad_direct = os.environ.get("FPL_GRAD_DIRECT", "1") != "0"
        self.wgrad_side_stream = False  # callers save / restore it; weight gradients run on the stream of their pass
        self._plans = {}
        self.grad_ready_hook = None     # callable(flat_grad, start, end, last) fired as buckets complete (DDP)
        self.grad_wait_hook = None      # callable() that makes the current stream wait for those all-reduces
        self.grad_bucket_bytes = 4 << 20
        self.grad_tail_bytes = 3 << 19      # 1.5 MB: the hand-over that cannot overlap anything stays below this
        self._master = None             # persistent flat gradient buffer (see _deliver_grads)
        self._head = UNet2D5_dsbn._HeadConv(self.out_conv)
        self._stem = None
        self._head_dirty = True
        self._stem_dirty = True
        self._build_units()

    # -- units ------------------------------------------------------------------------------
    def _build_units(self):
        for c in self.ft_chns:
            if c % 8 != 0:
                raise ValueError("feature_chns must be multiples of 8, got {0:}".format(self.ft_chns))
        blocks = [self.block0, self.block1, self.block2, self.block3, self.block4]
        ups = [self.up1, self.up2, self.up3, self.up4]
        self._down_units, self._up_units = [], []
        for i, b in enumerate(blocks):
            kd = 3 if b.dim == 3 else 1
            (c1, n1, r1, d1), (c2, n2, r2, _d2) = b.conv.units()
            self._down_units.append((_Unit("block%d.conv#1" % i, c1, n1, r1, d1, kd, is_stem=(i == 0)),
                                     _Unit("block%d.conv#2" % i, c2, n2, r2, None, kd)))
        for k, u in enumerate(ups, start=1):
            kd = 3 if u.dim == 3 else 1
            (c1, n1, r1, d1), (c2, n2, r2, _d2) = u.conv.units()
            self._up_units.append((_Unit("up%d.conv#1" % k, c1, n1, r1, d1, kd),
                                   _Unit("up%d.conv#2" % k, c2, n2, r2, None, kd)))
        # bilinear mode: the 1x1 projection in front of the up-sampling, one adapter per up block
        self._proj_units = []
        if self.bilinear:
            for k, u in enumerate(ups, start=1):
                conv = u.conv3d if u.dim == 3 else u.conv2d
                self._proj_units.append(_Unit("up%d.proj" % k, UNet2D5_dsbn._Conv1x1(conv), None, None, None, 1))

    class _HeadConv(object):
        """The head's weights zero-padded to 16 output channels (a plain tensor whose ``_version`` drives the
        weight-image cache), so that the (1,3,3) head runs through the same tensor-core kernels."""

        def __init__(self, out_conv):
            self.src = out_conv
            self.weight = None
            self.bias = None
            self.in_channels, self.out_channels = out_conv.in_channels, 16
            self.seen = None

        def sync(self, force):
            w = self.src.weight
            if self.weight is None or self.weight.device != w.device:
                self.weight = torch.zeros((16,) + tuple(w.shape[1:]), dtype=torch.float32, device=w.device)
                self.bias = torch.zeros(16, dtype=torch.float32, device=w.device)
                force = True
            ver = (w._version, self.src.bias._version)
            if force or ver != self.seen:
                k = w.shape[0]
                self.weight[:k].copy_(w.detach())
                self.bias[:k].copy_(self.src.bias.detach())
                self.seen = ver

    class _Conv1x1(object):
        """UpBlock's 1x1 conv of `bilinear=True` mode (unet2d5_dsbn.py:147-148,171,174) as a (1,3,3) conv whose off-centre
        taps are zero, so that forward / dgrad / wgrad run on the ordinary tensor-core conv kernels.  ``weight`` is a
        plain tensor kept in sync with the module (its ``_version`` drives the weight-image cache)."""

        def __init__(self, conv):
            self.src = conv
            self.weight = None
            self.in_channels, self.out_channels = conv.in_channels, conv.out_channels
            self.seen = None

        @property
        def bias(self):
            return self.src.bias

        def sync(self, force):
            w = self.src.weight
            co, ci = w.shape[0], w.shape[1]
            if self.weight is None or self.weight.device != w.device:
                self.weight = torch.zeros((co, ci, 1, 3, 3), dtype=torch.float32, device=w.device)
                force = True
            if force or w._version != self.seen:
                self.weight[:, :, 0, 1, 1].copy_(w.detach().reshape(co, ci))
                self.seen = w._version

    class _StemConv(object):
        """The 1-channel stem conv k(3,3,3) as a k(3,1,1) conv over the 16 "patch" channels written by
        fpl_patch9_c8 (channel kh*3+kw = in-plane neighbour): weight [Cout][16][3] kept in sync with the module."""

        def __init__(self, conv):
            self.src = conv
            self.weight = None
            self.seen = None
            self.image = None

        def sync(self, force):
            # K blocks [w_hi | w_hi | w_lo] against the A blocks [x_hi | x_lo | x_hi] of fpl_patch9_c8(split): the
            # stem stays fp32-accurate (x*w to ~2^-16) although every tensor-core operand is bf16
            w = self.src.weight
            co = w.shape[0]
            if self.weight is None or self.weight.device != w.device:
                self.weight = torch.zeros((co, 48, 3), dtype=torch.float32, device=w.device)
                self.image = torch.empty(48 * 3 * co, dtype=torch.bfloat16, device=w.device)
                force = True
            if force or w._version != self.seen:
                wk = w.detach()[:, 0].reshape(co, 3, 9).permute(0, 2, 1)
                hi = wk.to(torch.bfloat16).float()
                self.weight[:, 0:9, :].copy_(hi)
                self.weight[:, 16:25, :].copy_(hi)
                self.weight[:, 32:41, :].copy_(wk - hi)
                call("fpl_conv3d_k311_prep_weight", ptr(self.weight), 48, co, ptr(self.image), stream_ptr())
                self.seen = w._version

    def _grad_params(self, domain):
        """Parameters that receive gradients, in the order backward completes them."""
        out = [self.out_conv.weight, self.out_conv.bias]
        ups = [self.up1, self.up2, self.up3, self.up4]

        def unit_params(u):
            bn = u.dsbn.bns[domain]
            return [u.conv.weight, u.conv.bias, bn.weight, bn.bias, u.prelu.weight]

        for k in (3, 2, 1, 0):
            u1, u2 = self._up_units[k]
            out += unit_params(u2) + unit_params(u1)
            if self.bilinear:
                t = ups[k].conv3d if ups[k].dim == 3 else ups[k].conv2d
            else:
                t = ups[k].trans3d if ups[k].dim == 3 else ups[k].trans2d
            out += [t.weight, t.bias]
        for i in (4, 3, 2, 1, 0):
            u1, u2 = self._down_units[i]
            out += unit_params(u2) + unit_params(u1)
        return out

    # -- public forward ---------------------------------------------------------------------
    def forward_mc(self, x, domain_label, repeats, graph_lane=0):
        """K = ``repeats`` MC-dropout forwards of the SAME input in one call (no-grad): returns a list of K logits tensors,
        bit-identical to K consecutive ``forward`` calls (same seeds from torch's CPU generator), with the dropout-free
        encoder prefix computed once (agent_seg.py:897-911 runs K full passes; their first levels are identical)."""
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            raise RuntimeError("forward_mc is an inference call: wrap it in torch.no_grad()")
        if not 1 <= repeats <= self.kMaxMcRepeats:
            raise ValueError("repeats must be in [1, %d]" % self.kMaxMcRepeats)
        if repeats == 1:
            return [self.forward(x, domain_label, graph_lane)]
        return self.forward(x, domain_label, graph_lane, _repeats=repeats)

    def forward(self, x, domain_label=None, graph_lane=0, _repeats=1):
        """``graph_lane``: callers that run several no-grad forwards CONCURRENTLY on different streams (the
        Inferer's two half-batches) give each its own lane, i.e. its own captured graph and static buffers."""
        if domain_label is None:
            raise ValueError("UNet2D5_dsbn.forward needs domain_label")
        if x.dim() != 5:
            raise ValueError('expected 5D input (got {}D input)'.format(x.dim()))
        if not x.is_cuda:
            raise RuntimeError("fplplus_b200.UNet2D5_dsbn runs on CUDA (sm_100a) only; got a %s tensor" % x.device)
        domain = int(domain_label[0])
        if not 0 <= domain < self.num_domains:
            raise IndexError("domain_label %d out of range" % domain)
        x = x.float().contiguous()
        params = self._grad_params(domain)
        need_grad = torch.is_grad_enabled() and any(p.requires_grad for p in params)
        if need_grad:
            return _UNetFunction.apply(self, domain, x, *params)
        if self.cuda_graphs and not torch.cuda.is_current_stream_capturing():
            return self._forward_graphed(x, domain, graph_lane, _repeats)
        ws = self._infer_ws
        if ws is None or ws.device != x.device:
            ws = self._infer_ws = _Workspace(x.device)
        logits, _ = self._run_forward(x, domain, ws, _repeats)
        return logits

    # -- no-grad forwards replayed from CUDA graphs (sliding-window inference: 256 forwards / volume) --
    def _mode_signature(self, domain):
        sig = [self.training]
        for u1, u2 in self._down_units + self._up_units:
            for u in (u1, u2):
                sig.append(u.dsbn.bns[domain].training)
                if u.dropout is not None:
                    sig.append(u.dropout.training and u.dropout.p > 0.0)
        return tuple(sig)

    kMaxMcRepeats = 16      # seeds per graph lane: entry 0 is the ordinary dropout seed, 0..K-1 those of forward_mc

    def ensure_rng(self, device, lane=0):
        """The device-side dropout seed of a graph lane (must exist BEFORE a capture so that no allocation /
        zero-fill of it is recorded into the graph).  Lane 0 is also ``self._rng_dev`` (training graphs)."""
        t = self._rng_lanes.get(lane)
        if t is None or t.device != torch.device(device):
            t = self._rng_lanes[lane] = torch.zeros(self.kMaxMcRepeats, dtype=torch.int64, device=device)
        if lane == 0:
            self._rng_dev = t
        return t

    def _draw_seed(self):
        # torch's CPU generator, so torch.manual_seed makes MC-dropout passes reproducible
        return int(torch.empty((), dtype=torch.int64).random_().item()) & ((1 << 62) - 1)

    def _forward_graphed(self, x, domain, lane=0, repeats=1):
        key = (tuple(x.shape), domain, x.device.index, self._mode_signature(domain), lane, repeats)
        ent = self._graphs.get(key)
        if ent is None:
            # first sight of this (shape, domain, mode): run eagerly (also warms lazy driver state), capture next time
            self._graphs[key] = ent = {"graph": None, "calls": 0}
        ent["calls"] += 1
        if ent["graph"] is None and ent["calls"] < 2:
            ws = self._infer_wss.get(lane)
            if ws is None or ws.device != x.device:
                ws = self._infer_wss[lane] = _Workspace(x.device)
            logits, _ = self._run_forward(x, domain, ws, repeats)
            return logits
        rng = self.ensure_rng(x.device, lane)
        self.prepare(x.shape)                               # eager: a captured graph never restages weights
        if ent["graph"] is None:
            if len(self._graphs) > 24:                     # bound the memory held by stale shapes
                for k in [k for k in self._graphs if k != key][:8]:
                    del self._graphs[k]
            ent["x"] = x.clone()
            ent["ws"] = _Workspace(x.device)
            g = torch.cuda.CUDAGraph()
            self._seed_from_device, self._cur_lane = True, lane
            try:
                with torch.cuda.graph(g):
                    ent["out"], _ = self._run_forward(ent["x"], domain, ent["ws"], repeats)
            finally:
                self._seed_from_device, self._cur_lane = False, 0
            ent["graph"] = g
        ent["x"].copy_(x, non_blocking=True)
        if any(key[3][1:]) and self._dropout_masks is None:
            if repeats == 1:
                rng[0:1].fill_(self._draw_seed())
            else:
                for k in range(repeats):                   # the same draws, in the same order, as K separate forwards
                    rng[k:k + 1].fill_(self._draw_seed())
        ent["graph"].replay()
        if repeats > 1:
            return [o.clone() for o in ent["out"]]
        return ent["out"].clone()

    # -- helpers ----------------------------------------------------------------------------
    def _geometry(self, shape):
        n, c, d, h, w = shape
        if c != self.in_chns:
            raise ValueError("expected %d input channels, got %d" % (self.in_chns, c))
        geo = [(d, h, w)]
        for i in range(4):
            d, h, w = geo[-1]
            kd = 2 if self.dims[i] == 3 else 1
            if d % kd or h % 2 or w % 2:
                raise ValueError("input size %s is not divisible by the down-sampling factors" % (tuple(shape[2:]),))
            geo.append((d // kd, h // 2, w // 2))
        return geo

    def invalidate_weight_images(self):
        """Forget the staged bf16 weight images.  They are keyed on ``weight._version``, which every
        ordinary in-place update bumps (torch.optim's default implementations, ``load_state_dict``);
        optimisers that write through fused multi-tensor kernels (``Adam(fused=True)``) do not, so the
        agent calls this after ``optimizer.step()``."""
        for ent in self._img_cache.values():
            ent[0] = -1
        self._head_dirty = True
        self._stem_dirty = True

    # -- kernel plan ------------------------------------------------------------------------
    def _plan(self, n, geo, grad, sm100):
        """The kernel of every launch site of a forward (``grad``: and its backward) over ``n`` inputs with the level
        geometries ``geo`` (see _geometry), and the weight images those kernels read.  It depends on nothing else but
        the construction parameters and the library's image-size queries (no device work), so it is memoised."""
        key = (n, tuple(geo), bool(grad), bool(sm100))
        plan = self._plans.get(key)
        if plan is None:
            plan = self._plans[key] = self._make_plan(n, geo, grad, sm100)
        return plan

    def _make_plan(self, n, geo, grad, sm100):
        lib = ops._lib.load()
        impl_tc = self.conv_impl == "tc" and sm100
        ft, k_cls = self.ft_chns, self.n_class

        def tc(cin, cout):
            return impl_tc and cin % 16 == 0 and cout % 16 == 0

        def conv(cin, cout, kd, depth):
            if not tc(cin, cout):
                return "direct"
            # depth-folded tensor-core kernel (csrc/conv_tc_dfold.cu) for the small-channel k3 layers
            if kd == 3 and depth >= 2 and lib.fpl_conv3d_dfold_image_bytes(cin, cout) > 0:
                return "dfold"
            return "tc"

        plan = _Plan()
        plan.eval_fuse = self.eval_fuse and sm100
        # the 1-channel stem.  Training: "stem_direct" builds the 27-tap operand from the fp32 image in shared memory
        # (csrc/stem_tc.cu; 41 + 35 us against 81 + 40 us per forward + wgrad at 4x32x128x128, and no 134 MB patch
        # tensor kept until backward).  No-grad forwards keep "stem_patch" (fpl_patch9_c8 + a k(3,1,1) conv) whose
        # conv carries the activation in its epilogue.  "stem_cc": fpl_stem_conv_fwd for the other shapes.
        stem = self._down_units[0][0]
        d0, h0, w0 = geo[0]
        stem_tc = impl_tc and stem.cin == 1 and stem.kd == 3
        if grad and stem_tc and stem.cout == 16 and w0 >= 32 and h0 >= 4:
            plan.fwd[stem.name] = "stem_direct"
        elif stem_tc and d0 >= 2 and stem.cout in (16, 32, 64):
            plan.fwd[stem.name] = "stem_patch"
            plan.images.append(("stem", stem.conv, 0, 3))
        else:
            plan.fwd[stem.name] = "stem_cc"
        if grad:
            wg = plan.fwd[stem.name]
            if wg == "stem_cc" and tc(16, stem.cout) and stem.cin <= 8:
                wg = "stem_c8"          # the image packed into one zero-padded channel group, tensor-core wgrad
            plan.wgrad[stem.name] = wg
        units = [(u, geo[i][0]) for i in range(5) for u in self._down_units[i] if not u.is_stem]
        units += [(u, geo[3 - k][0]) for k in range(4) for u in self._up_units[k]]
        for u, depth in units:
            kern = plan.fwd[u.name] = conv(u.cin, u.cout, u.kd, depth)
            if kern != "direct":
                plan.images.append((kern, u.conv, 0, u.kd))
            if grad:
                kern = plan.dgrad[u.name] = conv(u.cout, u.cin, u.kd, depth)
                if kern != "direct":
                    plan.images.append((kern, u.conv, 1, u.kd))
                plan.wgrad[u.name] = "tapmajor" if sm100 and u.cin % 8 == 0 and u.cout % 16 == 0 else "direct"
        for k in range(4):
            c, c_low = ft[3 - k], ft[4 - k]
            if not self.bilinear:
                plan.up.append("tc" if tc(c_low, c) else "direct")
                continue
            if not tc(c_low, c):
                raise NotImplementedError("bilinear=True needs feature_chns that are multiples of 16 (tensor-core 1x1 "
                                          "projection)")
            plan.up.append("proj")
            pu = self._proj_units[k]
            plan.images += [("tc", pu.conv, t, 1) for t in ((0, 1) if grad else (0,))]
        if impl_tc and ft[0] in (16, 32) and k_cls <= 8 and d0 >= 2 and n * d0 <= 65535:
            plan.head = "cc"
        elif tc(ft[0], 16) and k_cls <= 8:
            plan.head = "tc"
        else:
            plan.head = "direct"
        # the images of the zero-padded head and of the tensor-core transposed convs are staged wherever those kernels
        # could run, also when this plan picks head.cu or bilinear up-sampling: unread there, but they only add
        # entries to the batched staging launches
        if tc(ft[0], 16) and k_cls <= 8:
            plan.images += [("tc", self._head, t, 1) for t in ((0, 1) if grad else (0,))]
        for up in (self.up1, self.up2, self.up3, self.up4):
            trans = up.trans3d if up.dim == 3 else up.trans2d
            if tc(trans.in_channels, trans.out_channels):
                plan.images += [("convt", trans, t, 2 if up.dim == 3 else 1) for t in ((0, 1) if grad else (0,))]
        return plan

    def prepare(self, shape, grad=False):
        """Stage every stale weight image that a forward (``grad``: and its backward) over inputs shaped ``shape``
        [N,C,D,H,W] reads, on the CURRENT stream, in batched launches; returns the pass's kernel plan.  Callers that fan
        passes out over several streams (the agent's two domain passes, the Inferer's two lanes) call this before the
        fork, so that no stream stages images while another reads them."""
        plan = self._plan(shape[0], self._geometry(tuple(shape)), grad, ops.is_sm100())
        lib = ops._lib.load()
        todo = {"dfold": [], "convt": [], "tc": []}
        synced = set()
        for kind, conv, t, kd in plan.images:
            if kind == "stem":
                if self._stem is None:
                    self._stem = UNet2D5_dsbn._StemConv(conv)
                self._stem.sync(self._stem_dirty)
                self._stem_dirty = False
                continue
            if hasattr(conv, "sync") and id(conv) not in synced:      # the padded head, the bilinear projections
                conv.sync(self._head_dirty)
                synced.add(id(conv))
            w = conv.weight
            key = (id(w), kind, t)
            ent = self._img_cache.get(key)
            if ent is None or ent[1].device != w.device:
                cin, cout = conv.in_channels, conv.out_channels
                if kind == "dfold":
                    nbytes = lib.fpl_conv3d_dfold_image_bytes(cout if t else cin, cin if t else cout)
                elif kind == "convt":
                    nbytes = lib.fpl_convt_weight_image_bytes(cin, cout, kd)
                else:
                    nbytes = lib.fpl_conv3d_weight_image_bytes(cout if t else cin, cin if t else cout, kd)
                ent = self._img_cache[key] = [-1, torch.empty(nbytes // 2, dtype=torch.bfloat16, device=w.device)]
            if ent[0] != w._version:
                todo[kind].append((w, conv.in_channels, conv.out_channels, kd, t, ent))
        self._head_dirty = False
        for kind, fn, cols, batch in (("dfold", "fpl_conv3d_dfold_prep_weight_batch", (1, 2, 4), 64),
                                      ("convt", "fpl_convt_prep_weight_batch", (1, 2, 3, 4), 16),
                                      ("tc", "fpl_conv3d_prep_weight_batch", (1, 2, 3, 4), 80)):
            for i in range(0, len(todo[kind]), batch):
                part = todo[kind][i:i + batch]
                m = len(part)
                arr_w = (ctypes.c_void_p * m)(*[e[0].data_ptr() for e in part])
                arr_img = (ctypes.c_void_p * m)(*[e[5][1].data_ptr() for e in part])
                ints = [(ctypes.c_int * m)(*[e[c] for e in part]) for c in cols]
                call(fn, m, arr_w, *ints, arr_img, stream_ptr())
                for e in part:
                    e[5][0] = e[0]._version
        return plan

    def _image(self, kind, conv, transpose=0):
        """A weight image staged by prepare() ("tc" / "dfold": transpose 1 = dgrad; "convt": mode 1 = dgrad)."""
        return self._img_cache[(id(conv.weight), kind, transpose)][1]

    def _conv_fwd(self, u, kern, xin, x_img, y, stats, n, geo, ws):
        d, h, w = geo
        st = stream_ptr()
        if kern == "stem_patch":
            xs = ws.c8("XS:stem", n, d, 32, h, w)
            call("fpl_patch9_c8", ptr(x_img), ptr(xs), 1, n, d, h, w, st)
            call("fpl_conv3d_tc_k311", ptr(xs), 4, 0, ptr(self._stem.image), ptr(u.conv.bias), ptr(y), y.shape[2], 0,
                 ptr(stats), n, d, h, w, 48, u.cout, 32, st)
        elif kern in ("stem_direct", "stem_cc"):
            call("fpl_stem_conv_fwd", ptr(x_img), ptr(u.conv.weight), ptr(u.conv.bias), ptr(y), y.shape[2], 0,
                 ptr(stats), n, u.cin, d, h, w, u.cout, u.kd, st)
        elif kern == "dfold":
            call("fpl_conv3d_tc_dfold", *xin.args(), ptr(self._image("dfold", u.conv)), ptr(u.conv.bias), ptr(y),
                 y.shape[2], 0, ptr(stats), n, d, h, w, u.cin, u.cout, st)
        elif kern == "tc":
            call("fpl_conv3d_tc", *xin.args(), ptr(self._image("tc", u.conv)), ptr(u.conv.bias), ptr(y), y.shape[2], 0,
                 ptr(stats), n, d, h, w, u.cin, u.cout, u.kd, st)
        else:
            call("fpl_conv3d_direct", *xin.args(), ptr(u.conv.weight), ptr(u.conv.bias), ptr(y), y.shape[2], 0,
                 ptr(stats), n, d, h, w, u.cin, u.cout, u.kd, 0, 0, st)

    def _eval_affine_refresh(self, domain, ws, plan):
        """Inference epilogue (csrc/common.cuh EpiAct): scale / shift of every conv unit whose BatchNorm is in eval mode,
        from the CURRENT running statistics, in one launch at the start of a no-grad forward (part of the captured
        graph, so replays follow the running statistics).  Returns {unit name: (scale, shift)}."""
        units = [u for pair in self._down_units + self._up_units for u in pair if not u.dsbn.bns[domain].training]
        if not units or not plan.eval_fuse:
            return {}
        key = "eval_affine:%d" % domain
        total = sum(2 * u.cout for u in units)
        buf = ws.get(key, (total,), torch.float32)
        out, o = {}, 0
        for u in units:
            out[u.name] = (buf[o:o + u.cout], buf[o + u.cout:o + 2 * u.cout])
            o += 2 * u.cout
        m = len(units)
        bns = [u.dsbn.bns[domain] for u in units]
        arr = lambda ts: (ctypes.c_void_p * m)(*[t.data_ptr() for t in ts])
        call("fpl_dsbn_eval_affine_batch", m, arr([b.weight for b in bns]), arr([b.bias for b in bns]),
             arr([b.running_mean for b in bns]), arr([b.running_var for b in bns]), arr([u.conv.bias for u in units]),
             arr([out[u.name][0] for u in units]), arr([out[u.name][1] for u in units]),
             (ctypes.c_int * m)(*[u.cout for u in units]), float(bns[0].eps), stream_ptr())
        return out

    def _unit_fwd_fused(self, u, kern, xin, x_img, out, aff, p, seed, offset, seed_dev, n, geo, ws):
        """Inference: conv with the eval-mode BatchNorm + PReLU (+ dropout) in its epilogue; writes the activation into
        ``out``.  Returns False when no fused kernel serves this unit (the caller runs the two-kernel path)."""
        d, h, w = geo
        st = stream_ptr()
        scale, shift = aff
        if kern == "stem_patch":
            if p > 0.0:
                return False
            xs = ws.c8("XS:stem", n, d, 32, h, w)
            call("fpl_patch9_c8", ptr(x_img), ptr(xs), 1, n, d, h, w, st)
            call("fpl_conv3d_tc_k311_act", ptr(xs), 4, 0, ptr(self._stem.image), *out.args(), n, d, h, w, 48, u.cout, 32,
                 ptr(scale), ptr(shift), ptr(u.prelu.weight), st)
            return True
        if kern == "dfold":
            if p > 0.0:
                return False
            call("fpl_conv3d_tc_dfold_act", *xin.args(), ptr(self._image("dfold", u.conv)), *out.args(), n, d, h, w,
                 u.cin, u.cout, ptr(scale), ptr(shift), ptr(u.prelu.weight), st)
            return True
        if kern == "tc":
            call("fpl_conv3d_tc_act", *xin.args(), ptr(self._image("tc", u.conv)), *out.args(), n, d, h, w, u.cin,
                 u.cout, u.kd, ptr(scale), ptr(shift), ptr(u.prelu.weight), p, seed, offset,
                 ptr(seed_dev) if p > 0.0 else None, st)
            return True
        return False

    def _unit_fwd(self, u, domain, xin, x_img, out, pooled, pool_idx, pool_kd, n, geo, ws, small, rec):
        """conv -> finalize -> act.  ``out``/``pooled`` are C8 views."""
        d, h, w = geo
        c = u.cout
        kern = rec["plan"].fwd[u.name]
        aff = rec["eval_affine"].get(u.name)
        if aff is not None:
            # no-grad forward, BatchNorm in eval mode: one kernel instead of two (dropout keeps the same Philox stream
            # positions as the two-kernel path)
            p, seed, offset = 0.0, 0, 0
            drop = u.dropout is not None and u.dropout.training and u.dropout.p > 0.0
            explicit = drop and self._dropout_masks is not None and u.name in self._dropout_masks
            if not explicit:
                if drop:
                    p, seed, offset = float(u.dropout.p), rec["seed"], rec["next_offset"]
                if self._unit_fwd_fused(u, kern, xin, x_img, out, aff, p, seed, offset, rec["seed_dev"], n, geo, ws):
                    if drop:
                        rec["next_offset"] += 2 * n * d * (c // 8) * h * w
                    if pooled is not None:
                        call("fpl_maxpool_c8", *out.args(), *pooled.args(), pool_kd, n, d, h, w, c, stream_ptr())
                    return
        y = ws.c8("Y:" + u.name, n, d, c, h, w)
        stats = small.f64(2 * c)
        self._conv_fwd(u, kern, xin, x_img, y, stats, n, geo, ws)
        bn = u.dsbn.bns[domain]
        if bn.weight.dtype != torch.float32:
            raise RuntimeError("fplplus_b200 supports tensor_type=float only")
        scale, shift, mean, invstd = small.f32(c), small.f32(c), small.f32(c), small.f32(c)
        training = 1 if bn.training else 0
        p, mask, seed, offset = 0.0, None, 0, 0
        if u.dropout is not None and u.dropout.training and u.dropout.p > 0.0:
            p = float(u.dropout.p)
            if self._dropout_masks is not None and u.name in self._dropout_masks:
                mask = self._dropout_masks[u.name]
            else:
                seed, offset = rec["seed"], rec["next_offset"]
                rec["next_offset"] += 2 * n * d * (c // 8) * h * w
        pv = pooled.args() if pooled is not None else (None, 0, 0)
        # statistics -> affine map (+ running statistics) in the prologue of the activation kernel
        call("fpl_dsbn_bn_act_fwd", ptr(y), ptr(stats), n * d * h * w, ptr(bn.weight), ptr(bn.bias),
             ptr(bn.running_mean), ptr(bn.running_var), ptr(bn.num_batches_tracked), float(bn.momentum), float(bn.eps),
             training, ptr(scale), ptr(shift), ptr(mean), ptr(invstd), ptr(u.prelu.weight), *out.args(), *pv,
             ptr(pool_idx), pool_kd, p, ptr(mask), seed, offset, ptr(rec["seed_dev"]) if p > 0.0 and mask is None else None,
             n, d, h, w, c, stream_ptr())
        rec[u.name] = dict(y=y, xin=xin, scale=scale, shift=shift, mean=mean, invstd=invstd, training=training,
                           p=p, mask=mask, seed=seed, offset=offset, geo=geo, bn=bn,
                           seed_dev=rec["seed_dev"] if p > 0.0 and mask is None else None)

    # -- whole-network forward --------------------------------------------------------------
    def _first_dropout_level(self):
        """Index of the first encoder level whose unit-1 dropout is active (5 = none): everything before it is
        deterministic, hence identical in all MC-dropout passes over the same input."""
        for i in range(5):
            dr = self._down_units[i][0].dropout
            if dr is not None and dr.training and dr.p > 0.0:
                return i
        return 5

    def _run_forward(self, x, domain, ws, repeats=1, grad=False):
        """``grad``: the forward of a training pass (its records feed _run_backward).  ``repeats`` > 1 (no-grad only):
        K MC-dropout passes over the same input in one call -- the encoder levels in front of the first active dropout
        run ONCE, the rest of the network K times with K dropout seeds; returns a list of K logits tensors
        (bit-identical to K separate forwards drawing the same seeds)."""
        n = x.shape[0]
        geo = self._geometry(x.shape)
        small = _SmallPool(ws, "fwd", x.device)
        plan = self.prepare(x.shape, grad)
        # dropout stream: (seed, per-layer offset) drawn from torch's CPU generator, so torch.manual_seed
        # makes MC-dropout passes reproducible; backward regenerates the same Philox stream
        if self._seed_from_device:
            seed, seed_dev = 0, self.ensure_rng(x.device, self._cur_lane)
        else:
            seed, seed_dev = self._draw_seed(), None
        rec = {"seed": seed, "seed_dev": seed_dev, "next_offset": 0, "geo": geo, "n": n, "x": x, "plan": plan}
        rec["eval_affine"] = {} if grad else self._eval_affine_refresh(domain, ws, plan)
        if repeats > 1:
            assert not torch.is_grad_enabled()
            seeds = [(seed, seed_dev if seed_dev is None else seed_dev[0:1])]
            for k in range(1, repeats):
                seeds.append((0, seed_dev[k:k + 1]) if self._seed_from_device else (self._draw_seed(), None))
            split = self._first_dropout_level()
            cur = None
            for i in range(split):
                cur = self._down_level(i, domain, cur, x, n, geo, ws, small, rec)
            outs = []
            for k in range(repeats):
                rec["seed"], rec["seed_dev"] = seeds[k]
                rec["next_offset"] = 0
                c2 = cur
                for i in range(split, 5):
                    c2 = self._down_level(i, domain, c2, x, n, geo, ws, small, rec)
                outs.append(self._up_path_and_head(c2, domain, x, n, geo, ws, small, rec)[0])
            return outs, rec
        cur = None
        for i in range(5):
            cur = self._down_level(i, domain, cur, x, n, geo, ws, small, rec)
        return self._up_path_and_head(cur, domain, x, n, geo, ws, small, rec)

    def _down_level(self, i, domain, cur, x, n, geo, ws, small, rec):
        ft = self.ft_chns
        u1, u2 = self._down_units[i]
        d, h, w = geo[i]
        c = ft[i]
        a1 = C8(ws.c8("A1:block%d" % i, n, d, c, h, w))
        self._unit_fwd(u1, domain, cur, x, a1, None, None, 0, n, geo[i], ws, small, rec)
        if i < 4:
            cat = ws.c8("cat%d" % i, n, d, 2 * c, h, w)
            d2, h2, w2 = geo[i + 1]
            pooled = C8(ws.c8("P%d" % i, n, d2, c, h2, w2))
            idx = ws.get("idx%d" % i, (n, d2, c // 8, h2, w2, 8), torch.uint8)
            pool_kd = 2 if self.dims[i] == 3 else 1
            self._unit_fwd(u2, domain, a1, None, C8(cat, 0, c), pooled, idx, pool_kd, n, geo[i], ws, small, rec)
            rec["idx%d" % i] = (idx, pool_kd)
            cur = pooled
        else:
            a2 = C8(ws.c8("A2:block4", n, d, c, h, w))
            self._unit_fwd(u2, domain, a1, None, a2, None, None, 0, n, geo[i], ws, small, rec)
            cur = a2
        return cur

    def _up_path_and_head(self, low, domain, x, n, geo, ws, small, rec):
        ft = self.ft_chns
        ups = [self.up1, self.up2, self.up3, self.up4]
        for k, lvl in zip(range(4), (3, 2, 1, 0)):
            up = ups[k]
            u1, u2 = self._up_units[k]
            d, h, w = geo[lvl]
            dl, hl, wl = geo[lvl + 1]
            c, c_low = ft[lvl], ft[lvl + 1]
            cat = ws.t["cat%d" % lvl]
            trans = up.trans3d if up.dim == 3 else up.trans2d
            kd2 = 2 if up.dim == 3 else 1
            kern = rec["plan"].up[k]
            if kern == "proj":
                # 1x1 projection at low resolution (a (1,3,3) conv with zero off-centre taps), then trilinear / bilinear
                # x2 up-sampling (align_corners=True) straight into the second half of the concat buffer
                pu = self._proj_units[k]
                t_low = ws.c8("T:up%d" % (k + 1), n, dl, c, hl, wl)
                call("fpl_conv3d_tc", *low.args(), ptr(self._image("tc", pu.conv)), ptr(pu.conv.bias), ptr(t_low),
                     c // 8, 0, None, n, dl, hl, wl, c_low, c, 1, stream_ptr())
                call("fpl_upsample2x_c8", ptr(t_low), c // 8, 0, ptr(cat), 2 * c // 8, c // 8, n, dl, hl, wl, c, kd2,
                     stream_ptr())
            elif kern == "tc":
                call("fpl_convt_k2s2_fwd_tc", *low.args(), ptr(self._image("convt", trans)), ptr(trans.bias), ptr(cat),
                     2 * c // 8, c // 8, n, dl, hl, wl, c_low, c, kd2, stream_ptr())
            else:
                call("fpl_convt_k2s2_fwd", *low.args(), ptr(trans.weight), ptr(trans.bias), ptr(cat), 2 * c // 8, c // 8,
                     n, dl, hl, wl, c_low, c, kd2, stream_ptr())
            rec["up%d.low" % (k + 1)] = low
            a1 = C8(ws.c8("A1:up%d" % (k + 1), n, d, c, h, w))
            self._unit_fwd(u1, domain, C8(cat, 0, 2 * c), None, a1, None, None, 0, n, geo[lvl], ws, small, rec)
            a2 = C8(ws.c8("A2:up%d" % (k + 1), n, d, c, h, w))
            self._unit_fwd(u2, domain, a1, None, a2, None, None, 0, n, geo[lvl], ws, small, rec)
            low = a2
        d, h, w = geo[0]
        logits = torch.empty((n, self.n_class, d, h, w), dtype=torch.float32, device=x.device)
        if rec["plan"].head == "cc":
            call("fpl_head_fwd", *low.args(), ptr(self.out_conv.weight), ptr(self.out_conv.bias), ptr(logits), n, d, h, w,
                 ft[0], self.n_class, stream_ptr())
        elif rec["plan"].head == "tc":
            call("fpl_head_conv_tc", *low.args(), ptr(self._image("tc", self._head)), ptr(self._head.bias), ptr(logits),
                 n, d, h, w, ft[0], self.n_class, stream_ptr())
        else:
            call("fpl_head_conv_fwd", *low.args(), ptr(self.out_conv.weight), ptr(self.out_conv.bias), ptr(logits),
                 n, d, h, w, ft[0], self.n_class, stream_ptr())
        rec["head_in"] = low
        return logits, rec

    # -- whole-network backward -------------------------------------------------------------
    def _unit_bwd(self, u, r, g1, g_pool, pool_idx, pool_kd, n, ws, small, grads, need_dx, fold, plan):
        """Backward of one conv unit.  Returns the C8 gradient wrt the unit's input (or None)."""
        d, h, w = r["geo"]
        c = u.cout
        st = stream_ptr()
        g1a = g1.args() if g1 is not None else (None, 0, 0)
        gpa = g_pool.args() if g_pool is not None else (None, 0, 0)
        common = (ptr(r["y"]), *g1a, *gpa, ptr(pool_idx), pool_kd, ptr(r["scale"]), ptr(r["shift"]), ptr(r["mean"]),
                  ptr(r["invstd"]), ptr(u.prelu.weight), r["p"], ptr(r["mask"]), r["seed"], r["offset"], ptr(r["seed_dev"]))
        red = small.f64(2 * c + 1)
        call("fpl_dsbn_act_bwd_reduce", *common, ptr(red), n, d, h, w, c, st)
        dy = ws.c8("dY:" + u.name, n, d, c, h, w)
        bn = r["bn"]
        call("fpl_dsbn_act_bwd_apply_fin", *common, ptr(red), r["training"], ptr(dy), n, d, h, w, c, st,
             ptr(grads[bn.weight]), ptr(grads[bn.bias]), ptr(grads[u.prelu.weight]), ptr(grads[u.conv.bias]))
        dw = grads[u.conv.weight]
        wgrad = plan.wgrad[u.name]
        if wgrad in ("stem_direct", "stem_cc"):
            call("fpl_stem_conv_wgrad", ptr(r["x_img"]), ptr(dy), c // 8, 0, ptr(dw), n, u.cin, d, h, w, c, u.kd, st)
            return None
        if wgrad == "stem_patch":
            # the patch tensor of the forward is still in the workspace: k(3,1,1) wgrad, one MMA per K step
            xs = ws.c8("XS:stem", n, d, 32, h, w)
            dw16 = ws.get("dW16s", (c, 16, 3), torch.float32)
            dw16.zero_()
            call("fpl_conv3d_wgrad_tc_k311", ptr(xs), 4, 0, ptr(dy), c // 8, 0, ptr(dw16), n, d, h, w, 16, c, st)   # hi half
            dw.view(c, 1, 3, 3, 3).add_(dw16[:, :9, :].permute(0, 2, 1).reshape(c, 1, 3, 3, 3))
            return None
        if wgrad == "stem_c8":
            # image -> one bf16 channel group (zero padded), then the tensor-core wgrad with Cin = 8
            x8 = ws.c8("X8", n, d, 8, h, w)
            call("fpl_pack_ncdhw_to_c8", ptr(r["x_img"]), u.cin, ptr(x8), 1, 0, 1, None, n, d, h, w, st)
            dw8 = ws.get("dW8", (c, 8, u.kd, 3, 3), torch.float32)
            dw8.zero_()
            call("fpl_conv3d_wgrad_tc", ptr(x8), 1, 0, ptr(dy), c // 8, 0, ptr(dw8), n, d, h, w, 8, c, u.kd, st)
            dw.view(c, u.cin, u.kd, 3, 3).add_(dw8[:, :u.cin])
            return None
        xin = r["xin"]
        if wgrad == "tapmajor":
            # tap-major scratch (coalesced epilogue atomics); folded into dw by one batched launch later
            scr = fold["alloc"](u.cout * u.cin * u.kd * 9)
            call("fpl_conv3d_wgrad_tc_tapmajor", *xin.args(), ptr(dy), u.cout // 8, 0, ptr(scr), n, d, h, w, u.cin,
                 u.cout, u.kd, st)
            fold["pending"].append((scr, dw, u.cout, u.cin, u.kd * 9))
        else:
            call("fpl_conv3d_wgrad", *xin.args(), ptr(dy), u.cout // 8, 0, ptr(dw), n, d, h, w, u.cin, u.cout, u.kd, st)
        if not need_dx:
            return None
        dx = ws.c8("dX:" + u.name, n, d, u.cin, h, w)
        kern = plan.dgrad[u.name]
        if kern == "dfold":
            call("fpl_conv3d_tc_dfold", ptr(dy), c // 8, 0, ptr(self._image("dfold", u.conv, 1)), None, ptr(dx),
                 u.cin // 8, 0, None, n, d, h, w, c, u.cin, st)
        elif kern == "tc":
            call("fpl_conv3d_tc", ptr(dy), c // 8, 0, ptr(self._image("tc", u.conv, 1)), None, ptr(dx), u.cin // 8, 0,
                 None, n, d, h, w, c, u.cin, u.kd, st)
        else:
            call("fpl_conv3d_direct", ptr(dy), c // 8, 0, ptr(u.conv.weight), None, ptr(dx), u.cin // 8, 0, None,
                 n, d, h, w, c, u.cin, u.kd, 1, 0, st)
        return C8(dx)

    def _run_backward(self, rec, dlogits, domain, ws):
        n, geo, ft, plan = rec["n"], rec["geo"], self.ft_chns, rec["plan"]
        params = self._grad_params(domain)
        sizes = [(p.numel() + 3) // 4 * 4 for p in params]
        flat = torch.zeros(sum(sizes), dtype=torch.float32, device=dlogits.device)
        grads, offs, o = {}, [], 0
        for p, s in zip(params, sizes):
            grads[p] = flat[o:o + p.numel()]
            offs.append(o)
            o += s
        fired = [0]
        # tap-major scratch of the conv weight gradients (one flat zeroed buffer per backward) + the list of layers
        # whose scratch still has to be folded into the PyTorch layout
        total = sum((u.conv.weight.numel() + 3) // 4 * 4 for pair in self._down_units + self._up_units for u in pair
                    if not u.is_stem) + 16 * self.ft_chns[0] * 9 + sum(
                        (t.weight.numel() + 3) // 4 * 4 for up in (self.up1, self.up2, self.up3, self.up4)
                        for t in (up.trans3d, up.trans2d) if t is not None) + sum(
                        9 * u.cin * u.cout for u in self._proj_units)
        scratch = ws.get("wgrad_scratch", (total,), torch.float32)
        scratch.zero_()
        cursor = [0]

        def alloc(numel):
            t = scratch[cursor[0]:cursor[0] + numel]
            cursor[0] += (numel + 3) // 4 * 4
            return t
        fold = {"alloc": alloc, "pending": []}

        def flush_fold():
            if not fold["pending"]:
                return
            part = fold["pending"]
            m = len(part)
            arr_s = (ctypes.c_void_p * m)(*[t[0].data_ptr() for t in part])
            arr_d = (ctypes.c_void_p * m)(*[t[1].data_ptr() for t in part])
            ints = [(ctypes.c_int * m)(*[t[k] for t in part]) for k in (2, 3, 4)]
            scout = (ctypes.c_int * m)(*[t[5] if len(t) > 5 else t[2] for t in part])
            call("fpl_wgrad_tapmajor_to_dw_batch", m, arr_s, arr_d, ints[0], ints[1], ints[2], scout, stream_ptr())
            fold["pending"] = []

        def fire(n_params_done):
            # gradients of params[:n_params_done] are final: hand the new flat range to the hook (DDP all-reduce)
            if self.grad_ready_hook is not None:
                end = offs[n_params_done - 1] + sizes[n_params_done - 1]
                last = n_params_done == len(params)
                # hand over >= grad_bucket_bytes at a time: every hand-over costs a fold launch and an all-reduce launch.
                # The all-reduce of the LAST hand-over has nothing left to hide under, so it is kept small: once less
                # than grad_tail_bytes remain, whatever has accumulated (>= 1 MB) goes out early.
                pending_b, remaining_b = (end - fired[0]) * 4, (len(flat) - end) * 4
                if end > fired[0] and (last or pending_b >= self.grad_bucket_bytes
                                       or (remaining_b <= self.grad_tail_bytes and pending_b >= (1 << 20))):
                    flush_fold()
                    self.grad_ready_hook(flat, fired[0], end, n_params_done == len(params))
                    fired[0] = end

        small = _SmallPool(ws, "bwd", dlogits.device)
        st = stream_ptr()
        d, h, w = geo[0]
        head_in = rec["head_in"]
        g = C8(ws.c8("dX:head", n, d, ft[0], h, w))
        dlogits = dlogits.contiguous()
        k = self.n_class
        if plan.head == "cc":
            # CUDA-core head dgrad (csrc/head.cu): one pass reads the fp32 logit gradient and writes the input gradient,
            # the one-channel-group bf16 copy the tensor-core wgrad consumes and the bias gradient
            dl8 = ws.c8("dL8", n, d, 8, h, w)
            call("fpl_head_dgrad", ptr(dlogits), ptr(self.out_conv.weight), *g.args(), ptr(dl8), 1, 0,
                 ptr(grads[self.out_conv.bias]), n, d, h, w, ft[0], k, st)
            scr = fold["alloc"](8 * ft[0] * 9)
            call("fpl_conv3d_wgrad_tc_tapmajor", *head_in.args(), ptr(dl8), 1, 0, ptr(scr), n, d, h, w, ft[0], 8, 1, st)
            fold["pending"].append((scr, grads[self.out_conv.weight], k, ft[0], 9, 8))
        elif plan.head == "tc":
            # dlogits -> bf16 C8-planar (zero padded to 16 channels) + the bias gradient; then the ordinary
            # tensor-core dgrad / wgrad with the padded head weights
            dl16 = ws.c8("dL16", n, d, 16, h, w)
            call("fpl_pack_ncdhw_to_c8", ptr(dlogits), k, ptr(dl16), 2, 0, 2, ptr(grads[self.out_conv.bias]), n, d, h, w, st)
            call("fpl_conv3d_tc", ptr(dl16), 2, 0, ptr(self._image("tc", self._head, 1)), None, *g.args(), None,
                 n, d, h, w, 16, ft[0], 1, st)
            # wgrad against the first channel group of dl16 only (classes padded to 8): 4 depth planes are stacked in
            # M and N, so one MMA set covers 4 planes (csrc/conv_wgrad_tc.cu, ndy = 4); only the k real classes are
            # folded into the head's gradient
            co = 8 if (ft[0] <= 32 and d >= 2) else 16
            scr = fold["alloc"](co * ft[0] * 9)
            call("fpl_conv3d_wgrad_tc_tapmajor", *head_in.args(), ptr(dl16), 2, 0, ptr(scr), n, d, h, w, ft[0], co, 1, st)
            fold["pending"].append((scr, grads[self.out_conv.weight], k, ft[0], 9, co))
        else:
            call("fpl_head_conv_bwd", *head_in.args(), ptr(self.out_conv.weight), ptr(dlogits), *g.args(),
                 ptr(grads[self.out_conv.weight]), ptr(grads[self.out_conv.bias]), n, d, h, w, ft[0], self.n_class, st)
        ups = [self.up1, self.up2, self.up3, self.up4]
        skip_grads = {}
        done = 2
        fire(done)
        for k, lvl in zip((3, 2, 1, 0), (0, 1, 2, 3)):
            u1, u2 = self._up_units[k]
            up = ups[k]
            c, c_low = ft[lvl], ft[lvl + 1]
            g = self._unit_bwd(u2, rec[u2.name], g, None, None, 0, n, ws, small, grads, True, fold, plan)
            # dgrad of unit 1 produces the gradient of the whole concat buffer; keep it alive per level
            dcat = self._unit_bwd(u1, rec[u1.name], g, None, None, 0, n, ws, small, grads, True, fold, plan)
            skip_grads[lvl] = C8(dcat.buf, 0, c)
            trans = up.trans3d if up.dim == 3 else up.trans2d
            kd2 = 2 if up.dim == 3 else 1
            dl, hl, wl = geo[lvl + 1]
            low = rec["up%d.low" % (k + 1)]
            glow = C8(ws.c8("dlow%d" % lvl, n, dl, c_low, hl, wl))
            if plan.up[k] == "proj":
                pu = self._proj_units[k]
                proj = up.conv3d if up.dim == 3 else up.conv2d
                g_t = ws.c8("dT:up%d" % (k + 1), n, dl, c, hl, wl)
                call("fpl_upsample2x_c8_bwd", ptr(dcat.buf), 2 * c // 8, c // 8, ptr(g_t), c // 8, 0, n, dl, hl, wl, c, kd2, st)
                call("fpl_channel_sum_c8", ptr(g_t), c // 8, 0, ptr(grads[proj.bias]), n, dl, hl, wl, c, st)
                # wgrad of the (1,3,3) stand-in: only its centre tap is the 1x1 weight
                scr = fold["alloc"](9 * c * c_low)
                call("fpl_conv3d_wgrad_tc_tapmajor", *low.args(), ptr(g_t), c // 8, 0, ptr(scr), n, dl, hl, wl, c_low, c, 1, st)
                fold["pending"].append((scr[4 * c * c_low:5 * c * c_low], grads[proj.weight], c, c_low, 1))
                call("fpl_conv3d_tc", ptr(g_t), c // 8, 0, ptr(self._image("tc", pu.conv, 1)), None, *glow.args(),
                     None, n, dl, hl, wl, c, c_low, 1, st)
            elif plan.up[k] == "tc":
                call("fpl_convt_k2s2_dgrad_tc", ptr(dcat.buf), 2 * c // 8, c // 8, ptr(self._image("convt", trans, 1)),
                     *glow.args(), n, dl, hl, wl, c_low, c, kd2, st)
                scr = fold["alloc"](c_low * c * 4 * kd2)
                call("fpl_convt_k2s2_wgrad_tc_tapmajor", *low.args(), ptr(dcat.buf), 2 * c // 8, c // 8, ptr(scr),
                     n, dl, hl, wl, c_low, c, kd2, st)
                fold["pending"].append((scr, grads[trans.weight], c, c_low, -4 * kd2))
                call("fpl_convt_k2s2_bwd", *low.args(), ptr(trans.weight), ptr(dcat.buf), 2 * c // 8, c // 8, None, 0, 0,
                     None, ptr(grads[trans.bias]), n, dl, hl, wl, c_low, c, kd2, st)       # bias gradient only
            else:
                call("fpl_convt_k2s2_bwd", *low.args(), ptr(trans.weight), ptr(dcat.buf), 2 * c // 8, c // 8, *glow.args(),
                     ptr(grads[trans.weight]), ptr(grads[trans.bias]), n, dl, hl, wl, c_low, c, kd2, st)
            g = glow
            done += 12
            fire(done)
        g_pool = None
        for i in (4, 3, 2, 1, 0):
            u1, u2 = self._down_units[i]
            r1 = rec[u1.name]
            if i == 4:
                g = self._unit_bwd(u2, rec[u2.name], g, None, None, 0, n, ws, small, grads, True, fold, plan)
            else:
                idx, pool_kd = rec["idx%d" % i]
                g = self._unit_bwd(u2, rec[u2.name], skip_grads[i], g_pool, idx, pool_kd, n, ws, small, grads, True, fold,
                                   plan)
            r1["x_img"] = rec["x"]
            if i > 0:
                g_pool = self._unit_bwd(u1, r1, g, None, None, 0, n, ws, small, grads, True, fold, plan)
            else:
                self._unit_bwd(u1, r1, g, None, None, 0, n, ws, small, grads, False, fold, plan)
            done += 10
            fire(done)
        assert done == len(params)
        flush_fold()
        return self._deliver_grads(params, offs, flat, grads)

    # -- gradient delivery --------------------------------------------------------------------
    def _master_grads(self, device):
        """Persistent flat fp32 buffer behind every p.grad (all parameters that can receive gradients, both domains),
        plus one device-resident segment table per domain for fpl_grad_scatter_add."""
        m = self._master
        if m is None or m["buf"].device != device:
            order, off, o = [], {}, 0
            for d in range(self.num_domains):
                for p in self._grad_params(d):
                    if p not in off:
                        off[p] = o
                        order.append(p)
                        o += (p.numel() + 3) // 4 * 4
            m = self._master = {"buf": torch.zeros(o, dtype=torch.float32, device=device), "off": off, "tables": {},
                                "event": None}
        return m

    def _deliver_grads(self, params, offs, flat, grads):
        """Hands one backward pass's gradients to the optimiser.  Default: ONE fpl_grad_scatter_add launch adds the
        pass's flat buffer into the master buffer and p.grad is a view of that buffer (autograd gets None: its ~65
        per-parameter AccumulateGrad adds for the second domain pass disappear).  The first pass after a
        zero_grad(set_to_none=True) zeroes the master buffer.  FPL_GRAD_DIRECT=0 (read at construction), or a p.grad that
        is not ours, falls back to returning the gradients to autograd."""
        views = [grads[p].view(p.shape) for p in params]
        if not self.grad_direct:
            return views
        m = self._master_grads(flat.device)
        base, off = m["buf"].data_ptr(), m["off"]
        if any(p.grad is not None and p.grad.data_ptr() != base + 4 * off[p] for p in params):
            return views
        if self.grad_wait_hook is not None:
            self.grad_wait_hook()                     # DDP: the asynchronous all-reduces of `flat` must have landed
        cur = torch.cuda.current_stream()
        capturing = torch.cuda.is_current_stream_capturing()
        if self.out_conv.weight.grad is None:
            m["buf"].zero_()
            m["event"] = torch.cuda.Event()
            m["event"].record(cur)
            m["event_captured"] = capturing
        elif m["event"] is not None and m.get("event_captured", False) == capturing:
            # the other pass's stream may have issued the zeroing (an event recorded inside a graph capture cannot be
            # waited on from eager work; eager work after a replay is ordered by its stream anyway)
            cur.wait_event(m["event"])
        key = tuple(id(p) for p in params)
        tab = m["tables"].get(key)
        if tab is None:
            rows = [[so, off[p], p.numel()] for p, so in zip(params, offs)]
            tab = m["tables"][key] = (torch.tensor(rows, dtype=torch.int32, device=flat.device),
                                      max(p.numel() for p in params))
        call("fpl_grad_scatter_add", ptr(m["buf"]), ptr(flat), ptr(tab[0]), len(params), tab[1], stream_ptr())
        for p in params:
            if p.grad is None:
                p.grad = m["buf"][off[p]:off[p] + p.numel()].view(p.shape)
        return [None] * len(params)


class _SmallPool(object):
    """Bump allocator for per-layer fp32/fp64 scratch (statistics, scale/shift, reductions): one
    zero-fill per pass instead of one per layer."""

    def __init__(self, ws, tag, device, n32=1 << 16, n64=1 << 15):
        self.b32 = ws.get("small32:" + tag, (n32,), torch.float32)
        self.b64 = ws.get("small64:" + tag, (n64,), torch.float64)
        self.b32.zero_()
        self.b64.zero_()
        self.o32 = self.o64 = 0

    def f32(self, n):
        n4 = (n + 3) // 4 * 4
        t = self.b32[self.o32:self.o32 + n]
        self.o32 += n4
        assert self.o32 <= self.b32.numel()
        return t

    def f64(self, n):
        n2 = (n + 1) // 2 * 2
        t = self.b64[self.o64:self.o64 + n]
        self.o64 += n2
        assert self.o64 <= self.b64.numel()
        return t


class _UNetFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, net, domain, x, *params):
        if torch.cuda.is_current_stream_capturing():
            # buffers baked into a CUDA graph: a private workspace (allocated from the graph's pool) that is
            # parked in _graph_ws_keep instead of going back to the recycling pool
            ws, home = _Workspace(x.device), net._graph_ws_keep
        else:
            ws, home = (net._pool.pop() if net._pool else _Workspace(x.device)), net._pool
            if ws.device != x.device:
                ws = _Workspace(x.device)
        logits, rec = net._run_forward(x, domain, ws, grad=True)
        ctx.net, ctx.domain, ctx.rec = net, domain, rec
        ctx.lease = _Lease(home, ws)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        net = ctx.net
        grads = net._run_backward(ctx.rec, dlogits, ctx.domain, ctx.lease.ws)
        ctx.rec = None
        return (None, None, None) + tuple(grads)
