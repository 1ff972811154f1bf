"""Host-side train/test agent of the hot path, mirroring PyMIC's ``net_run_dsbn`` plugin surface
(reference: PyMIC/pymic/net_run_dsbn/agent_abstract.py:28-357, agent_seg.py:35-1065,
util/parse_config.py:70-111, net_run/get_optimizer.py:9-57).

Same names, same ``.cfg`` keys, same call order:

* ``parse_config`` / ``synchronize_config``                      (util/parse_config.py:86-111)
* ``SegmentationAgent(config, stage)`` with the plugin setters ``set_net_dict / set_loss_dict /
  set_network / set_inferer / set_optimizer / set_scheduler / set_datasets``
  (agent_abstract.py:67-134), ``create_network`` (agent_seg.py:82-105), ``create_optimizer``
  (agent_abstract.py:320-337), ``create_loss_calculator`` (agent_seg.py:113-132),
  ``get_loss_value`` (:134-142), ``training_all`` (:415-508), ``validation`` (:509-604),
  ``train_valid`` (:689-831, same checkpoint dict / ``_latest.txt`` / ``_best.txt``), ``infer``
  (:834-964, plain pseudo-label branch and the FPL branch with K=6 MC-dropout passes) and ``run``.

What is different underneath (B200-first, SURVEY.md §8):

* one process per GPU (``torchrun``): gradients of each backward are all-reduced over NCCL in
  buckets that overlap the rest of the backward (``GradAllReducer``); inference shards volumes
  round-robin over ranks with no communication except the final gather of ~100 scalars;
* the train loop never synchronises per step: loss and hard-Dice counters accumulate on the
  device and are read once per ``training_all`` round (the reference does 2 ``.item()``/``.cpu()``
  syncs per step, agent_seg.py:476,495);
* the FPL statistics / pseudo labels / agreement weights stay on the device (csrc/filter.cu); only
  the uint8 label volume or two scalars per volume come back to the host;
* the CPU transform pipeline is replaced: without ``set_loaders`` / ``set_datasets``, a training
  run builds one ``DevicePatchSampler`` per domain from ``[dataset] {1,2}_train_csv`` and
  ``train_transform`` (datapath.py: volumes resident in HBM, RandomCrop / RandomFlip /
  NormalizeWithMeanStd per step on the device); otherwise loaders are any iterables of batch dicts,
  validation and test loaders always so; ``NpyVolumeDataset`` is the minimal built-in for ``.npy``
  / ``.nii`` volumes.

As in the reference only ``training_all`` semantics train (``training()`` of the shipped
``dual=False`` cfgs has no ``backward()``; SURVEY.md §3.1): ``dual`` is accepted and both values
run the optimiser step.
"""
import configparser
import copy
import logging
import os
import time

import numpy as np
import torch
import torch.nn as nn
from torch.optim import lr_scheduler

from . import fpl
from .inferer import Inferer
from .loss import CombinedLoss, hard_dice_from_sums
from .registry import loss_dict as _default_loss_dict
from .registry import net_dict as _default_net_dict


# ------------------------------------------------------------------------------------------
# .cfg parsing (util/parse_config.py:7-111): INI, keys lower-cased, values type-sniffed
# ------------------------------------------------------------------------------------------
def _is_int(s):
    body = s[1:] if s[:1] == '-' else s
    return all('0' <= ch <= '9' for ch in body)


def _is_float(s):
    for sep in ('.', 'e'):
        if sep in s:
            parts = s.split(sep)
            if sep == '.' and './' in s:
                return False
            if sep == 'e' and s[0] == 'e':
                continue
            return len(parts) == 2 and _is_int(parts[0]) and _is_int(parts[1])
    return False


def _scalar(s):
    if _is_int(s):
        return int(s)
    if _is_float(s):
        return float(s)
    if s.lower() in ('true', 'false'):
        return s.lower() == 'true'
    if s.lower() == 'none':
        return None
    return s


def parse_value_from_string(val_str):
    if _is_int(val_str):
        return int(val_str)
    if _is_float(val_str):
        return float(val_str)
    if val_str[0] == '[' and val_str[-1] == ']':
        return [_scalar(item.strip()) for item in val_str[1:-1].split(',')]
    return _scalar(val_str)


def parse_config(filename):
    cp = configparser.ConfigParser()
    cp.read(filename)
    out = {}
    for section in cp.sections():
        out[section] = {}
        for key in cp[section]:
            val = str(cp[section][key])
            if len(val) > 0:
                out[section][key] = parse_value_from_string(val)
    return out


def synchronize_config(config):
    config['dataset']['labeltoprobability_class_num'] = config['network']['class_num']
    if 'PartialLabelToProbability' in (config['dataset'].get('train_transform') or []):
        config['dataset']['partiallabeltoprobability_class_num'] = config['network']['class_num']
    return config


def seed_torch(seed=1):
    """agent_abstract.py:13-26 (cudnn flags are irrelevant here: no cuDNN on the path)."""
    import random
    random.seed(seed)
    os.environ['PYTHONHASHSEED'] = str(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
    if torch.cuda.is_available():
        torch.cuda.manual_seed(seed)


def keyword_match(a, b):
    return a.lower() == b.lower()


def get_optimizer(name, net_params, optim_params, capturable=False):
    """net_run/get_optimizer.py:9-36 (the optimisers FPL+ configs select; coupled-L2 Adam).
    ``capturable``: Adam keeps its step counter and learning rate on the device so that the whole
    optimiser step can live inside a CUDA graph."""
    lr = optim_params['learning_rate']
    momentum = optim_params.get('momentum', 0.9)
    weight_decay = optim_params.get('weight_decay', 0.0)
    if keyword_match(name, "SGD"):
        return torch.optim.SGD(net_params, lr, momentum=momentum, weight_decay=weight_decay)
    if keyword_match(name, "Adam"):
        params = list(net_params)
        # same update rule (coupled L2, per-parameter step counters, torch's state_dict layout) as ONE launch of the
        # library's multi-tensor kernel (optim.FusedAdam, csrc/adam.cu); CPU parameters keep torch's implementation
        if len(params) > 0 and all(p.is_cuda for p in params):
            from .optim import FusedAdam
            if capturable:
                lr = torch.tensor(float(lr), dtype=torch.float32, device=params[0].device)
            return FusedAdam(params, lr, weight_decay=weight_decay)
        return torch.optim.Adam(params, lr, weight_decay=weight_decay)
    if keyword_match(name, "RMSprop"):
        return torch.optim.RMSprop(net_params, lr, momentum=momentum, weight_decay=weight_decay)
    raise ValueError("unsupported optimizer {0:}".format(name))


def get_lr_scheduler(optimizer, sched_params):
    """net_run/get_optimizer.py:39-57."""
    name = sched_params.get("lr_scheduler")
    if name is None:
        return None
    lr_gamma = sched_params["lr_gamma"]
    if keyword_match(name, "ReduceLROnPlateau"):
        patience = sched_params["reducelronplateau_patience"] / sched_params["iter_valid"]
        return lr_scheduler.ReduceLROnPlateau(optimizer, mode="max", factor=lr_gamma, patience=patience)
    if keyword_match(name, "MultiStepLR"):
        return lr_scheduler.MultiStepLR(optimizer, sched_params["lr_milestones"], lr_gamma,
                                        sched_params.get("last_iter", -1))
    raise ValueError("unsupported lr scheduler {0:}".format(name))


# ------------------------------------------------------------------------------------------
# multi-GPU plumbing: one process per GPU, NCCL (gloo on CPU tests)
# ------------------------------------------------------------------------------------------
def dist_info():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


class GradAllReducer(object):
    """Averages gradients over ranks while backward is still running.

    ``UNet2D5_dsbn`` writes all gradients of one backward into ONE flat fp32 buffer in the order
    backward completes them and calls ``grad_ready_hook(flat, start, end)`` whenever a further
    prefix is final.  Ranges are coalesced into buckets of >= ``bucket_bytes`` and all-reduced
    asynchronously (NCCL runs them on its own stream, NVLS over NVSwitch when available), so the
    22.6 MB of gradients travel under the remaining backward kernels; ``finish`` waits for the
    outstanding handles and applies the 1/world scale.  Parameters without gradients (2-D twins,
    1x1 convs, the other domain's BN) are never touched: no unused-parameter search."""

    def __init__(self, bucket_bytes=0, group=None):
        # bucket_bytes = 0: every range the network hands over is reduced at once (UNet2D5_dsbn already coalesces its
        # hand-overs to >= grad_bucket_bytes and keeps the LAST one small, see net.py fire())
        self.bucket_bytes = bucket_bytes
        self.group = group
        self._pending = []
        self._start = None

    def hook(self, flat, start, end, last=False):
        import torch.distributed as dist
        if self._start is None:
            self._start = start
        if (end - self._start) * 4 >= self.bucket_bytes or last:
            seg = flat[self._start:end]
            if seg.is_cuda:
                # NCCL averages inside the collective: no separate 1/world scaling kernel per bucket
                self._pending.append(dist.all_reduce(seg, op=dist.ReduceOp.AVG, group=self.group, async_op=True))
            else:                   # gloo (CPU tests) has no AVG
                seg.mul_(1.0 / dist.get_world_size(self.group))
                self._pending.append(dist.all_reduce(seg, op=dist.ReduceOp.SUM, group=self.group, async_op=True))
            self._start = None

    def finish(self):
        for h in self._pending:
            h.wait()
        self._pending = []
        self._start = None


class DeferredGradAllReducer(object):
    """ONE all-reduce per optimiser step, after both domain passes: the master gradient buffer behind every ``p.grad``
    (``UNet2D5_dsbn._deliver_grads``: both passes of ``training_all`` are scatter-added into it) is averaged over the
    ranks in a single NCCL call just before the optimiser update.

    Against ``GradAllReducer`` (bucketed all-reduces of EACH pass's flat buffer under the remaining backward kernels)
    this moves half the bytes (the two domain passes share every conv weight: 22.6 MB once instead of twice), needs no
    per-bucket fold launches, and no NCCL kernel runs while the one-CTA-per-SM persistent conv kernels do (measured in
    round 2: every weight-gradient launch ~10 us slower under a concurrent all-reduce, +0.4 ms per step at 8 GPUs for
    a ~0.1 ms collective).  The cost is that the collective is exposed; profiles/README.md has the A/B."""

    def __init__(self, net, group=None):
        self.net, self.group = net, group

    def _reduce(self, t):
        import torch.distributed as dist
        if t.is_cuda:
            dist.all_reduce(t, op=dist.ReduceOp.AVG, group=self.group)
        else:                       # gloo (CPU tests) has no AVG
            t.mul_(1.0 / dist.get_world_size(self.group))
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)

    def finish(self):
        m = getattr(self.net, "_master", None)
        grads = [p.grad for p in self.net.parameters() if p.grad is not None]
        if not grads:
            return
        if m is not None:
            lo, hi = m["buf"].data_ptr(), m["buf"].data_ptr() + 4 * m["buf"].numel()
            if all(lo <= g.data_ptr() < hi for g in grads):
                self._reduce(m["buf"])
                return
        for g in grads:             # gradients delivered through autograd (FPL_GRAD_DIRECT=0, foreign p.grad)
            self._reduce(g)


def reserve_sms_for_nccl(ctas=None, sm_budget=None):
    """Data-parallel runs: how the SMs are shared between NCCL's all-reduce kernels (which overlap backward) and the
    library's persistent one-CTA-per-SM kernels.  Call BEFORE ``init_process_group`` (NCCL reads NCCL_MAX_CTAS when the
    communicator is created).

    ``ctas`` ($FPL_NCCL_CTAS, default 0 = leave NCCL alone) caps NCCL's CTAs; ``sm_budget`` ($FPL_SM_BUDGET, default 148
    minus the cap) is the SM count every persistent grid is sized for (fpl_set_sm_budget).  Measured on 8 B200
    (profiles/README.md): capping NCCL slows the all-reduce more than the freed SMs gain (5.06 ms uncapped, 5.15 at
    16 CTAs / 132 SMs, 5.31 at 8 / 140), so the default leaves both alone; the knobs stay for other topologies."""
    if ctas is None:
        ctas = int(os.environ.get("FPL_NCCL_CTAS", "0"))
    if ctas > 0:
        os.environ.setdefault("NCCL_MAX_CTAS", str(ctas))
        os.environ.setdefault("NCCL_MIN_CTAS", str(min(ctas, 4)))
    held = int(os.environ.get("NCCL_MAX_CTAS", "0") or 0)
    if sm_budget is None:
        sm_budget = int(os.environ.get("FPL_SM_BUDGET", 148 - held))
    if sm_budget != 148:
        from . import lib as _lib
        _lib.call("fpl_set_sm_budget", int(sm_budget))
    return held


def shard_round_robin(items, rank, world):
    """Volumes are independent (agent_seg.py:881 loop): rank r takes items r, r+world, ..."""
    return [it for i, it in enumerate(items) if i % world == rank]


# ------------------------------------------------------------------------------------------
# minimal built-in dataset (file formats are out of scope; this covers .npy volumes)
# ------------------------------------------------------------------------------------------
class NpyVolumeDataset(torch.utils.data.Dataset):
    """Rows of (image[, label[, pixel_weight[, image_weight]]]) file names (.npy, or .nii / .nii.gz through
    artefacts.py -- the 4 columns of config_dual/data_vs/train_vs_t1s_wi+wp.csv) -> the batch-dict keys
    the agent consumes (io/nifty_dataset.py:171-218): 'image' [C,D,H,W] fp32, 'label_prob'
    [class,D,H,W] fp32, 'pixel_weight' [1,D,H,W] folded by set_weight_ (:165-168), 'image_weight',
    'names'."""

    def __init__(self, rows, class_num, root_dir=""):
        self.rows, self.class_num, self.root = rows, class_num, root_dir

    def __len__(self):
        return len(self.rows)

    def _load(self, rel):
        from . import artefacts
        return artefacts.load_volume(os.path.join(self.root, rel))

    def __getitem__(self, i):
        row = self.rows[i]
        img = np.asarray(self._load(row[0])).astype(np.float32)
        if img.ndim == 3:
            img = img[None]
        sample = {'image': torch.from_numpy(img), 'names': row[0]}
        if len(row) > 1 and row[1]:
            lab = np.asarray(self._load(row[1]))
            sample['label_prob'] = torch.from_numpy(
                np.stack([lab == c for c in range(self.class_num)], 0).astype(np.float32))
        if len(row) > 2 and row[2]:
            w = np.asarray(self._load(row[2])).astype(np.float32)[None]
            iw = float(row[3]) if len(row) > 3 else 1.0
            w = np.where(w < 1, 0, w).astype(np.float32) * np.float32(iw)      # set_weight_
            sample['pixel_weight'] = torch.from_numpy(w)
            sample['image_weight'] = iw
        return sample


# ------------------------------------------------------------------------------------------
# the agent
# ------------------------------------------------------------------------------------------
class SegmentationAgent(object):
    def __init__(self, config, stage='train'):
        assert stage in ['train', 'inference', 'test']
        self.config = config
        self.stage = 'test' if stage == 'inference' else stage
        self.train_set = self.valid_set = self.test_set = None
        self.net = self.optimizer = self.scheduler = None
        self.net_dict, self.loss_dict = _default_net_dict, _default_loss_dict
        self.inferer = None
        self.loss_calculator = None
        self.train_loaders = [None, None]
        self.valid_loaders = [None, None]
        self.test_loader = None
        self.tensor_type = config.get('dataset', {}).get('tensor_type', 'float')
        self.deterministic = config.get('training', {}).get('deterministic', True)
        self.random_seed = config.get('training', {}).get('random_seed', 1)
        if self.deterministic:
            seed_torch(self.random_seed)
        if self.tensor_type != 'float':
            raise ValueError("fplplus_b200 supports tensor_type = float only (bf16 tensor-core path)")
        self.rank, self.world = dist_info()
        self.device = None
        self.reducer = None
        self.fpl_uda = config.get('training', {}).get('train_fpl_uda', False)
        self.glob_it = 0
        self.last_outputs = {}
        # B200-first: the whole optimiser step (both forwards, loss, backward, gradient all-reduce, Adam)
        # is captured once per batch signature into a CUDA graph and replayed ([training] cuda_graph, default on)
        self.use_cuda_graph = (bool(config.get('training', {}).get('cuda_graph', True))
                               and os.environ.get("FPL_CUDA_GRAPH", "1") != "0")
        self._graphs = {}
        self._host_it = 0
        self.dual_stream = (bool(config.get('training', {}).get('dual_stream', True))
                            and os.environ.get("FPL_DUAL_STREAM", "1") != "0")
        self._side_stream = None
        self._copy_stream = None
        if self.dual_stream:
            try:
                torch.autograd.graph.set_warn_on_accumulate_grad_stream_mismatch(False)
            except Exception:
                pass

    # -- plugin setters (agent_abstract.py:67-134) -------------------------------------------
    def set_datasets(self, train_set, valid_set, test_set):
        self.train_set, self.valid_set, self.test_set = train_set, valid_set, test_set

    def set_loaders(self, train=None, valid=None, test=None):
        """train / valid: a loader or a [domain-1 loader, domain-2 loader] pair."""
        def pair(x):
            if x is None:
                return [None, None]
            return list(x) if isinstance(x, (list, tuple)) else [x, None]
        if train is not None:
            self.train_loaders = pair(train)
        if valid is not None:
            self.valid_loaders = pair(valid)
        if test is not None:
            self.test_loader = test

    def set_network(self, net):
        self.net = net

    def set_net_dict(self, net_dict):
        self.net_dict = net_dict

    def set_loss_dict(self, loss_dict):
        self.loss_dict = loss_dict

    def set_optimizer(self, optimizer):
        self.optimizer = optimizer

    def set_scheduler(self, scheduler):
        self.scheduler = scheduler

    def set_inferer(self, inferer):
        self.inferer = inferer

    # -- construction --------------------------------------------------------------------------
    def _pick_device(self, section):
        if not torch.cuda.is_available():
            raise RuntimeError("fplplus_b200 runs on CUDA (sm_100a) only: no GPU visible")
        if self.world > 1:
            dev = int(os.environ.get("LOCAL_RANK", self.rank))
        else:
            gpus = self.config.get(section, {}).get('gpus', [0])
            dev = gpus[0] if isinstance(gpus, (list, tuple)) else int(gpus)
        torch.cuda.set_device(dev)
        self.device = torch.device("cuda:{0:}".format(dev))
        return self.device

    def create_dataset(self):
        """agent_abstract.py:241-318: loaders come from set_loaders(), or are wrapped around the
        datasets given to set_datasets() with the cfg's batch sizes.  With neither, the training loaders are
        ``DevicePatchSampler``s built from ``[dataset] {1,2}_train_csv`` and ``train_transform``
        (``datapath.samplers_from_config``): the volumes stay on the training GPU."""
        ds = self.config.get('dataset', {})
        bs = ds.get('train_batch_size', 1)
        if self.stage == 'train':
            if (self.train_loaders[0] is None and self.train_set is None
                    and (ds.get('1_train_csv') or ds.get('2_train_csv'))):
                from .datapath import samplers_from_config
                self.train_loaders = samplers_from_config(self.config, self._pick_device('training'), self.rank,
                                                          self.world)
            if self.train_loaders[0] is None and self.train_set is not None:
                sets = self.train_set if isinstance(self.train_set, (list, tuple)) else [self.train_set]

                def train_loader(s):
                    if self.world > 1:
                        # one process per GPU: every rank draws a disjoint shard of each epoch's permutation
                        sampler = torch.utils.data.distributed.DistributedSampler(
                            s, num_replicas=self.world, rank=self.rank, shuffle=True, seed=int(self.random_seed),
                            drop_last=True)
                        return torch.utils.data.DataLoader(s, batch_size=bs, sampler=sampler, drop_last=True)
                    return torch.utils.data.DataLoader(s, batch_size=bs, shuffle=True, drop_last=True)
                self.train_loaders = [train_loader(s) for s in sets] + [None] * (2 - len(sets))
            if self.valid_loaders[0] is None and self.valid_set is not None:
                sets = self.valid_set if isinstance(self.valid_set, (list, tuple)) else [self.valid_set]
                self.valid_loaders = [torch.utils.data.DataLoader(s, batch_size=1, shuffle=False) for s in sets] \
                    + [None] * (2 - len(sets))
        elif self.test_loader is None and self.test_set is not None:
            self.test_loader = torch.utils.data.DataLoader(self.test_set, batch_size=1, shuffle=False)

    def create_network(self):
        if self.net is None:
            net_name = self.config['network']['net_type']
            if net_name not in self.net_dict:
                raise ValueError("Undefined network {0:}".format(net_name))
            self.net = self.net_dict[net_name](self.config['network'])
        self.net.float()
        n = sum(p.numel() for p in self.net.parameters() if p.requires_grad)
        logging.info('parameter number {0:}'.format(n))

    def get_parameters_to_update(self):
        return self.net.parameters()

    def create_optimizer(self, params):
        opt_params = self.config['training']
        if self.optimizer is None:
            self._graph_capable = (self.use_cuda_graph and keyword_match(opt_params['optimizer'], "Adam")
                                   and opt_params.get("lr_scheduler") in (None, "MultiStepLR"))
            self.optimizer = get_optimizer(opt_params['optimizer'], params, opt_params, capturable=self._graph_capable)
        last_iter = -1
        if getattr(self, 'checkpoint', None) is not None:
            self.optimizer.load_state_dict(self.checkpoint['optimizer_state_dict'])
            last_iter = self.checkpoint['iteration'] - 1
            if getattr(self, "_graph_capable", False):
                # a checkpoint written by torch.optim.Adam carries a float learning rate: the captured step reads it
                # from device memory
                for gph in self.optimizer.param_groups:
                    if not torch.is_tensor(gph['lr']):
                        gph['lr'] = torch.tensor(float(gph['lr']), dtype=torch.float32, device=gph['params'][0].device)
        self._host_it = last_iter + 1
        if self.scheduler is None:
            opt_params["last_iter"] = last_iter
            if getattr(self, "_graph_capable", False):
                # the learning rate lives in a device tensor read by the captured Adam: MultiStepLR is evaluated
                # in closed form on the host (get_optimizer.py:50-54) and written into that tensor when it changes
                self.scheduler = None
                self._lr_base = float(opt_params['learning_rate'])
                self._lr_now = None
                self._set_lr(self._lr_at(self._host_it))
            else:
                self.scheduler = get_lr_scheduler(self.optimizer, opt_params)

    def create_loss_calculator(self):
        loss_name = self.config['training']['loss_type']
        if isinstance(loss_name, (list, tuple)):
            self.loss_calculator = CombinedLoss(self.config['training'], self.loss_dict)
        elif loss_name not in self.loss_dict:
            raise ValueError("Undefined loss function {0:}".format(loss_name))
        else:
            self.loss_calculator = self.loss_dict[loss_name](self.config['training'])

    def get_loss_value(self, data, pred, gt, fpl_uda=False):
        loss_input_dict = {'prediction': pred, 'ground_truth': gt}
        if fpl_uda and data.get('pixel_weight', None) is not None:
            pw = data['pixel_weight']
            loss_input_dict['pixel_weight'] = pw.to(pred.device, non_blocking=True)
            if data.get('image_weight', None) is not None:
                loss_input_dict['image_weight'] = data['image_weight']
                # device data path: a uint8 agreement code (0/1/2 = 0/0.5/1) is NOT yet folded with the image weight;
                # the loss kernel applies NiftyDataset.set_weight_ (io/nifty_dataset.py:165-168) per voxel
                loss_input_dict['fold_image_weight'] = pw.dtype == torch.uint8
        return self.loss_calculator(loss_input_dict)

    # -- one optimiser step (agent_seg.py:459-495) -------------------------------------------
    def _to_device(self, t):
        if torch.is_tensor(t) and t.dtype == torch.uint8:       # label maps / agreement codes stay 1 byte per voxel
            return t.to(self.device, non_blocking=True)
        return torch.as_tensor(t).to(self.device, dtype=torch.float32, non_blocking=True)

    @staticmethod
    def _truth_key(data):
        """'label_prob' (fp32 one-hot/soft, the PyMIC batch layout) or 'label' (uint8 label map, device data path)."""
        return 'label_prob' if data.get('label_prob', None) is not None else 'label'

    def _lr_at(self, it):
        tr = self.config['training']
        if tr.get("lr_scheduler") is None:
            return self._lr_base
        n = sum(1 for m in tr["lr_milestones"] if m <= it)
        return self._lr_base * (tr["lr_gamma"] ** n)

    def _set_lr(self, lr):
        if self._lr_now is None or lr != self._lr_now:
            for gph in self.optimizer.param_groups:
                if torch.is_tensor(gph['lr']):
                    gph['lr'].fill_(lr)
                else:
                    gph['lr'] = lr
            self._lr_now = lr

    def current_lr(self):
        lr = self.optimizer.param_groups[0]['lr']
        return self._lr_now if torch.is_tensor(lr) else lr

    def enable_data_parallel(self, mode=None, group=None):
        """Gradient averaging over the ranks of ``torch.distributed`` (one process per GPU; agent_seg.py:695 wraps the
        net in nn.DataParallel instead).  ``mode`` ([training] grad_allreduce / $FPL_GRAD_ALLREDUCE): 'deferred'
        (default) = one all-reduce of the master gradient buffer per step, 'overlapped' = bucketed all-reduces of each
        domain pass under its backward (round 1)."""
        if mode is None:
            mode = os.environ.get("FPL_GRAD_ALLREDUCE", self.config.get('training', {}).get('grad_allreduce', 'deferred'))
        if mode == 'overlapped':
            self.reducer = GradAllReducer(group=group)
            self.net.grad_ready_hook = self.reducer.hook
            self.net.grad_wait_hook = self.reducer.finish
        elif mode == 'deferred':
            self.reducer = DeferredGradAllReducer(self.net, group=group)
            self.net.grad_ready_hook = self.net.grad_wait_hook = None
        else:
            raise ValueError("grad_allreduce must be 'deferred' or 'overlapped', got %r" % (mode,))
        return self.reducer

    def _step_body(self, batches):
        """forward(s) + loss + backward (+ overlapped gradient all-reduce) + optimiser update; device work only."""
        inval = getattr(self.net, "invalidate_weight_images", None)
        if inval is not None:
            inval()                 # fused optimisers do not bump tensor versions (see UNet2D5_dsbn)
        present = [d for d, b in enumerate(batches) if b is not None]
        main = torch.cuda.current_stream()
        fork = self.dual_stream and len(present) == 2
        if fork:
            # the two domain passes are independent until the optimiser: run them on two streams so that the
            # tensor-pipe-bound convolutions of one overlap the HBM-bound BatchNorm/activation kernels of the other
            # (autograd replays each backward on the stream its forward ran on)
            # every weight image both passes read is staged here, once, before the fork: a pass that staged one
            # after the fork would race the other stream's reads
            prepare = getattr(self.net, "prepare", None)
            if prepare is not None:
                for d in present:
                    prepare(tuple(batches[d]['image'].shape), grad=True)
            if self._side_stream is None:
                self._side_stream = torch.cuda.Stream()
            self._side_stream.wait_stream(main)
        losses, dices = [], []
        for d in present:
            data = batches[d]
            stream = self._side_stream if (fork and d == present[1]) else main
            with torch.cuda.stream(stream):
                x = self._to_device(data['image'])
                y = self._to_device(data[self._truth_key(data)])
                out = self.net(x, domain_label=d * torch.ones(x.shape[0], dtype=torch.long))
                loss_d = self.get_loss_value(data, out, y, self.fpl_uda)
                hd = getattr(self.loss_calculator, "last_hard_dice", None)
                dices.append(hd() if hd is not None else None)
            if fork and stream is not main:
                main.wait_stream(stream)
            losses.append(loss_d)
        n_dom = len(losses)
        # L = mean_d L_d (agent_seg.py:467).  (Making every domain loss its own backward root with a constant upstream
        # gradient, so that no scalar kernels sit between forward and backward, measured neutral and moved the reported
        # value's two kernels into the tail of the step: not kept.)
        loss = losses[0] if n_dom == 1 else (losses[0] + losses[1]) / n_dom if n_dom == 2 else sum(losses) / n_dom
        loss.backward()
        if fork:
            main.wait_stream(self._side_stream)
        if self.reducer is not None:
            self.reducer.finish()
        self.optimizer.step()
        if inval is not None:
            inval()                 # the staged images now lag the updated masters (validation / infer re-stage)
        return loss.detach(), dices

    def train_step(self, batches):
        """zero_grad; for each domain d present: L_d = loss(net(x_d, d), y_d[, w_d]); L = mean_d L_d;
        backward (gradient all-reduce overlapped when world > 1); optimizer.step; scheduler.step.
        ``batches``: list indexed by domain of batch dicts (host or device tensors) or None.
        Returns (loss tensor on the device, [hard-Dice tensor per domain]) -- no host sync.
        With ``cuda_graph`` the device work of the step is replayed from a captured graph; the returned
        tensors are then static buffers that the next step overwrites."""
        if getattr(self, "_graph_capable", False) and self.use_cuda_graph:
            out = self._train_step_graphed(batches)
            self._host_it += 1
            self._set_lr(self._lr_at(self._host_it))
            return out
        self.optimizer.zero_grad(set_to_none=True)
        out = self._step_body(batches)
        self._host_it += 1
        if self.scheduler is not None and not isinstance(self.scheduler, lr_scheduler.ReduceLROnPlateau):
            self.scheduler.step()
        elif getattr(self, "_graph_capable", False):
            self._set_lr(self._lr_at(self._host_it))
        return out

    _TENSOR_KEYS = ('image', 'label_prob', 'label', 'pixel_weight', 'image_weight')
    _WEIGHT_KEYS = ('pixel_weight', 'image_weight')

    def _graph_keys(self, b):
        """Tensor entries of a batch dict that the captured step reads (static buffers refreshed before every replay)."""
        keys = []
        for k in self._TENSOR_KEYS:
            v = b.get(k, None)
            if v is None or (k in self._WEIGHT_KEYS and not self.fpl_uda):
                continue
            if k == 'label' and b.get('label_prob', None) is not None:
                continue
            if k == 'image_weight' and not (torch.is_tensor(v) and b.get('pixel_weight', None) is not None
                                            and b['pixel_weight'].dtype == torch.uint8):
                continue                    # already folded into an fp32 pixel_weight by the loader: the loss ignores it
            keys.append(k)
        return keys

    def _train_step_graphed(self, batches):
        key = tuple(None if b is None else tuple((k, tuple(b[k].shape), str(b[k].dtype)) for k in self._graph_keys(b))
                    for b in batches)
        ent = self._graphs.get(key)
        if ent is None:
            ent = self._graphs[key] = {"graph": None, "calls": 0}
        ent["calls"] += 1
        if ent["graph"] is None and ent["calls"] <= 3:
            # eager warm-up steps: optimiser state, workspaces, lazy driver state
            self.optimizer.zero_grad(set_to_none=True)
            return self._step_body(batches)
        if ent["graph"] is None:
            static = []
            for b in batches:
                if b is None:
                    static.append(None)
                    continue
                sb = {k: self._to_device(b[k]).clone() for k in self._graph_keys(b)}
                static.append(sb)
            ent["static"] = static
            if hasattr(self.net, "ensure_rng"):
                self.net.ensure_rng(self.device)
            self.net._seed_from_device = True
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            self.optimizer.zero_grad(set_to_none=True)
            try:
                with torch.cuda.graph(g):
                    ent["out"] = self._step_body(static)
            finally:
                self.net._seed_from_device = False
            ent["graph"] = g
            # the capture itself does not execute: fall through to the first replay with this step's data
        # inputs -> the graph's static buffers.  Host batches go through a double-buffered staging area filled by
        # a copy stream, so the H2D transfer of step i runs under the replay of step i-1; the hand-over into the
        # static buffers is a device-to-device copy on the compute stream.
        main = torch.cuda.current_stream()
        on_host = any(b is not None and any(not b[k].is_cuda for k in self._TENSOR_KEYS if k in sb)
                      for b, sb in zip(batches, ent["static"]))
        if on_host:
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream()
            if "staging" not in ent:
                ent["staging"] = [[None if sb is None else {k: torch.empty_like(v) for k, v in sb.items() if torch.is_tensor(v)}
                                   for sb in ent["static"]] for _ in range(2)]
                ent["stg_free"] = [torch.cuda.Event(), torch.cuda.Event()]
                for ev in ent["stg_free"]:
                    ev.record(main)
            slot = ent["calls"] & 1
            stg = ent["staging"][slot]
            cs = self._copy_stream
            cs.wait_event(ent["stg_free"][slot])
            with torch.cuda.stream(cs):
                for b, st_ in zip(batches, stg):
                    if b is None:
                        continue
                    for k in self._TENSOR_KEYS:
                        if k in st_:
                            st_[k].copy_(b[k], non_blocking=True)
                arrived = torch.cuda.Event()
                arrived.record(cs)
            main.wait_event(arrived)
            for st_, sb in zip(stg, ent["static"]):
                if sb is None:
                    continue
                for k in self._TENSOR_KEYS:
                    if k in sb:
                        sb[k].copy_(st_[k], non_blocking=True)
            ent["stg_free"][slot].record(main)
        else:
            for b, sb in zip(batches, ent["static"]):
                if b is None:
                    continue
                for k in self._TENSOR_KEYS:
                    if k in sb:
                        sb[k].copy_(b[k], non_blocking=True)
        if getattr(self.net, "_rng_dev", None) is not None:
            self.net._rng_dev.fill_(self.net._draw_seed())
        ent["graph"].replay()
        inval = getattr(self.net, "invalidate_weight_images", None)
        if inval is not None:
            # the replay updated the fp32 masters after staging: a no-grad forward that follows (validation, infer)
            # must not trust the host-side "fresh" marks set while the graph was captured
            inval()
        return ent["out"]

    def _next(self, d, iters):
        try:
            return next(iters[d])
        except StopIteration:
            iters[d] = iter(self.train_loaders[d])
            return next(iters[d])

    def training_all(self):
        iter_valid = self.config['training']['iter_valid']
        n_dom = self.config['network']['num_domains']
        self.net.train()
        iters = [iter(self.train_loaders[d]) if self.train_loaders[d] is not None else None for d in range(2)]
        loss_acc = torch.zeros((), dtype=torch.float32, device=self.device)
        dice_acc = [None] * n_dom
        for _it in range(iter_valid):
            batches = [self._next(d, iters) if (d < n_dom and iters[d] is not None) else None for d in range(2)]
            loss, dices = self.train_step(batches)
            loss_acc += loss
            k = 0
            for d, b in enumerate(batches):
                if b is None:
                    continue
                if dices[k] is not None:
                    dice_acc[d] = dices[k].clone() if dice_acc[d] is None else dice_acc[d] + dices[k]
                k += 1
        # ONE device->host read per round
        train_avg_loss = float(loss_acc) / iter_valid / int(n_dom)
        cls = [(a / iter_valid).cpu().numpy() for a in dice_acc if a is not None]
        cls_dice = np.mean(np.stack(cls, 0), 0) if cls else np.zeros(self.config['network']['class_num'])
        return {'loss': train_avg_loss, 'avg_dice': float(cls_dice.mean()), 'class_dice': cls_dice}

    training = training_all     # SURVEY.md §3.1: the shipped training() never calls backward()

    def validation(self):
        class_num = self.config['network']['class_num']
        n_dom = self.config['network']['num_domains']
        if self.inferer is None:
            infer_cfg = dict(self.config.get('testing', {}))
            infer_cfg['class_num'] = class_num
            self.inferer = Inferer(infer_cfg)
        res = []
        self._broadcast_state(buffers_only=True)
        hold = getattr(self.loss_calculator, "last", None)
        exact = hold.pop("sums_allreduce", None) if isinstance(hold, dict) else None     # every rank validates ALL volumes
        self.net.eval()
        with torch.no_grad():
            for d in range(n_dom):
                losses, dices = [], []
                loader = self.valid_loaders[d]
                for data in (loader if loader is not None else []):
                    x, y = self._to_device(data['image']), self._to_device(data[self._truth_key(data)])
                    out = self.inferer.run(self.net, x, domain_label=d * torch.ones(x.shape[0], dtype=torch.long))
                    losses.append(self.get_loss_value(data, out, y))
                    for i in range(x.shape[0]):        # per-volume hard Dice (agent_seg.py:541-545)
                        self.get_loss_value(data, out[i:i + 1].contiguous(), y[i:i + 1].contiguous())
                        dices.append(self.loss_calculator.last_hard_dice())
                if losses:
                    res.append((torch.stack(losses).mean(), torch.stack(dices).mean(0)))
        self.net.train()
        if exact is not None:
            hold["sums_allreduce"] = exact
        if not res:
            return {'loss': 0.0, 'avg_dice': 0.0, 'class_dice': np.zeros(class_num)}
        host = [(float(l), c.cpu().numpy()) for l, c in res]
        tr = self.config['training']
        if tr.get('val_t2', False) and len(host) > 1:
            pick = [host[1]]
        elif tr.get('val_t1', False):
            pick = [host[0]]
        else:
            pick = host
        loss = float(np.mean([h[0] for h in pick]))
        cls = np.mean(np.stack([h[1] for h in pick], 0), 0)
        scal = self._agree_scalars({'loss': loss, 'avg_dice': float(cls.mean()), 'class_dice': cls})
        if isinstance(self.scheduler, lr_scheduler.ReduceLROnPlateau):
            self.scheduler.step(scal['avg_dice'])
        return scal

    # -- train/valid driver with the reference's checkpoint protocol (agent_seg.py:689-831) ----
    def _ckpt_names(self):
        ckpt_dir = self.config['training']['ckpt_save_dir']
        prefix = self.config['training'].get('ckpt_prefix', None)
        if prefix is None:
            prefix = ckpt_dir.split('/')[-1]
        return ckpt_dir, prefix

    def train_valid(self):
        tr = self.config['training']
        self.dual = tr.get('dual', True)
        self.fpl_uda = tr.get('train_fpl_uda', False)
        self._pick_device('training')
        self.net.to(self.device)
        if self.world > 1:
            if os.environ.get("NCCL_MAX_CTAS") or os.environ.get("FPL_SM_BUDGET"):
                reserve_sms_for_nccl()                 # the communicator exists already: only the grid budget applies
            self.enable_data_parallel()
        ckpt_dir, prefix = self._ckpt_names()
        iter_start, iter_max, iter_valid = tr['iter_start'], tr['iter_max'], tr['iter_valid']
        iter_save = tr.get('iter_save', None)
        early_stop_it = tr.get('early_stop_patience', None)
        if iter_save is None:
            iter_save_list = [iter_max]
        elif isinstance(iter_save, (tuple, list)):
            iter_save_list = iter_save
        else:
            iter_save_list = range(0, iter_max + 1, iter_save)
        self.max_val_dice, self.max_val_it, self.best_model_wts, self.checkpoint = 0.0, 0, None, None
        if iter_start > 0:
            name = "{0:}/{1:}_{2:}.pt".format(ckpt_dir, prefix, iter_start)
            self.checkpoint = torch.load(name, map_location=self.device, weights_only=False)
            self.checkpoint['valid_pred'] = 0
            self.net.load_state_dict(self.checkpoint['model_state_dict'])
            self.max_val_it = iter_start
            self.best_model_wts = self.checkpoint['model_state_dict']
        self._broadcast_state()
        self.create_optimizer(self.get_parameters_to_update())
        self.create_loss_calculator()
        self._install_exact_dp_dice()
        if self.rank == 0:
            os.makedirs(ckpt_dir, exist_ok=True)
        self.glob_it = iter_start
        history = []
        for it in range(iter_start, iter_max, iter_valid):
            lr_value = self.current_lr() if hasattr(self, '_lr_now') else self.optimizer.param_groups[0]['lr']
            t0 = time.time()
            train_scalars = self.training_all()
            t1 = time.time()
            valid_scalars = self.validation()
            t2 = time.time()
            self.glob_it = it + iter_valid
            logging.info("it {0:} lr {1:} train loss {2:.4f} dice {3:.4f} | valid loss {4:.4f} dice {5:.4f} | "
                         "{6:.2f}s/{7:.2f}s".format(self.glob_it, lr_value, train_scalars['loss'],
                                                    train_scalars['avg_dice'], valid_scalars['loss'],
                                                    valid_scalars['avg_dice'], t1 - t0, t2 - t1))
            history.append((self.glob_it, train_scalars, valid_scalars))
            if valid_scalars['avg_dice'] > self.max_val_dice or self.best_model_wts is None:
                self.max_val_dice = valid_scalars['avg_dice']
                self.max_val_it = self.glob_it
                self.best_model_wts = copy.deepcopy(self.net.state_dict())
            stop_now = early_stop_it is not None and self.glob_it - self.max_val_it > early_stop_it
            if (self.glob_it in iter_save_list or stop_now) and self.rank == 0:
                torch.save({'iteration': self.glob_it, 'valid_pred': valid_scalars['avg_dice'],
                            'model_state_dict': self.net.state_dict(),
                            'optimizer_state_dict': self.optimizer.state_dict()},
                           "{0:}/{1:}_{2:}.pt".format(ckpt_dir, prefix, self.glob_it))
                with open("{0:}/{1:}_latest.txt".format(ckpt_dir, prefix), 'wt') as f:
                    f.write(str(self.glob_it))
            if stop_now:
                logging.info("The training is early stopped")
                break
        if self.rank == 0:
            torch.save({'iteration': self.max_val_it, 'valid_pred': self.max_val_dice,
                        'model_state_dict': self.best_model_wts,
                        'optimizer_state_dict': self.optimizer.state_dict()},
                       "{0:}/{1:}_{2:}.pt".format(ckpt_dir, prefix, self.max_val_it))
            with open("{0:}/{1:}_best.txt".format(ckpt_dir, prefix), 'wt') as f:
                f.write(str(self.max_val_it))
        return history

    def get_checkpoint_name(self):
        ckpt_mode = self.config['testing']['ckpt_mode']
        if ckpt_mode in (0, 1):
            ckpt_dir, prefix = self._ckpt_names()
            txt = ckpt_dir + '/' + prefix + ("_latest.txt" if ckpt_mode == 0 else "_best.txt")
            with open(txt, 'r') as f:
                it_num = f.read().replace('\n', '')
            return "{0:}/{1:}_{2:}.pt".format(ckpt_dir, prefix, it_num)
        return self.config['testing']['ckpt_name']

    # -- inference / pseudo labels / FPL image weights (agent_seg.py:834-964) -------------------
    def infer(self, load_checkpoint=True):
        te = self.config['testing']
        domain = te['domian_label']                 # (sic) the reference's key
        self.FPL = te.get('fpl', False)
        device = self._pick_device('testing')
        self.net.to(device)
        if te.get('evaluation_mode', True):
            self.net.eval()
            if te.get('test_time_dropout', False) or self.FPL:
                def test_time_dropout(m):
                    if type(m) == nn.Dropout:
                        m.train()
                self.net.apply(test_time_dropout)
        if load_checkpoint:
            ckpt_name = self.get_checkpoint_name()
            if isinstance(ckpt_name, (tuple, list)):
                raise ValueError("ckpt_mode 3 (multi-checkpoint ensemble) is outside the hot path")
            checkpoint = torch.load(ckpt_name, map_location=device, weights_only=False)
            self.net.load_state_dict(checkpoint['model_state_dict'])
        if self.inferer is None:
            infer_cfg = dict(te)
            infer_cfg['class_num'] = self.config['network']['class_num']
            self.inferer = Inferer(infer_cfg)
        k_passes = int(te.get('fpl_mc_passes', 6))  # hard-coded 6 in the reference (:898)
        if self.FPL and not 1 <= k_passes <= fpl.max_mc_passes():
            raise ValueError("fpl_mc_passes = %d not in [1, %d]" % (k_passes, fpl.max_mc_passes()))
        uncertainty_list, pending = {}, []
        outputs = {}
        volumes = list(self.test_loader)
        with torch.no_grad():
            for data in shard_round_robin(volumes, self.rank, self.world):
                images = self._to_device(data['image'])
                names = data['names']
                name = names[0] if isinstance(names, (list, tuple)) else names
                dl = domain * torch.ones(images.shape[0], dtype=torch.long)
                if self.FPL:
                    # the K MC-dropout passes in one sweep: their dropout-free encoder levels are computed once
                    if k_passes > 1 and hasattr(self.net, "forward_mc") and isinstance(self.inferer, Inferer):
                        passes = self.inferer.run(self.net, images, dl, mc_passes=k_passes)
                    else:
                        passes = [self.inferer.run(self.net, images, domain_label=dl) for _ in range(k_passes)]
                    stats, _ = fpl.mc_uncertainty(passes)
                    pending.append((name, stats))          # stays on the device until the loop ends
                else:
                    pred = self.inferer.run(self.net, images, domain_label=dl)
                    outputs[name] = fpl.pseudo_label(pred)
        if self.FPL:
            for name, stats in pending:
                uncertainty_list[name] = [fpl.finish_uncertainty(stats)]
            uncertainty_list = self._gather_dict(uncertainty_list)
            srt = fpl.sort_uncertainty(uncertainty_list)
            path = te.get('fpl_uncertainty_sorted', None)
            if path and self.rank == 0:
                np.save(path, np.asarray(srt, dtype=object))
            self.last_outputs = {'uncertainty_sorted': srt}
            return srt
        self.last_outputs = {k: v.cpu().numpy() for k, v in outputs.items()}
        self.save_outputs(self.last_outputs)
        return self.last_outputs

    # -- multi-process agreement (one process per GPU) ------------------------------------------
    def _broadcast_state(self, buffers_only=False):
        """Rank 0's parameters / buffers on every rank.  Parameters: once, before the first step (ranks may have been
        initialised from different seeds).  Buffers (BatchNorm running statistics, rank-local under data parallelism):
        before every validation, which reproduces nn.DataParallel, whose replica 0 shares its buffers with the wrapped
        module (agent_seg.py:695) -- and makes the validation score, hence early stopping / ReduceLROnPlateau /
        best-model choice, identical on all ranks."""
        if self.world == 1:
            return
        import torch.distributed as dist
        tensors = list(self.net.buffers()) if buffers_only else list(self.net.parameters()) + list(self.net.buffers())
        for dtype in sorted({t.dtype for t in tensors}, key=str):
            group = [t for t in tensors if t.dtype == dtype]
            flat = torch.cat([t.detach().reshape(-1) for t in group])
            dist.broadcast(flat, src=0)
            o = 0
            with torch.no_grad():
                for t in group:
                    t.copy_(flat[o:o + t.numel()].view_as(t))
                    o += t.numel()
        inval = getattr(self.net, "invalidate_weight_images", None)
        if inval is not None and not buffers_only:
            inval()

    def _install_exact_dp_dice(self):
        """[training] exact_dp_dice = True (SURVEY 8e, optional): nn.DataParallel (agent_seg.py:695) evaluates Dice / CE over
        the gathered GLOBAL batch (loss/seg/dice.py:29-35); one process per GPU evaluates them per rank, which is a
        different gradient because Dice is a ratio of sums.  With this key the (6C+3) partial sums of the fused loss
        are all-reduced between its reduce and gradient passes (120 bytes per domain pass), which restores the
        reference's multi-GPU loss exactly; the default keeps the per-rank loss (no extra collective)."""
        hold = getattr(self.loss_calculator, "last", None)
        if self.world == 1 or hold is None or not self.config['training'].get('exact_dp_dice', False):
            return
        import torch.distributed as dist
        world = self.world

        def allreduce(sums):
            dist.all_reduce(sums, op=dist.ReduceOp.SUM)
            return world
        hold["sums_allreduce"] = allreduce

    def _agree_scalars(self, scal):
        """Rank 0's validation scalars on every rank (bit-identical control flow: stop_now, scheduler, best model)."""
        if self.world == 1:
            return scal
        import torch.distributed as dist
        cls = np.asarray(scal['class_dice'], np.float64)
        t = torch.tensor([scal['loss'], scal['avg_dice']] + cls.tolist(), dtype=torch.float64, device=self.device)
        dist.broadcast(t, src=0)
        v = t.tolist()
        return {'loss': v[0], 'avg_dice': v[1], 'class_dice': np.asarray(v[2:], cls.dtype).reshape(cls.shape)}

    def _gather_dict(self, d):
        if self.world == 1:
            return d
        import torch.distributed as dist
        parts = [None] * self.world
        dist.all_gather_object(parts, d)
        merged = {}
        for p in parts:
            merged.update(p)
        return merged

    def save_outputs(self, outputs):
        """uint8 label volumes -> ``output_dir/<name>`` (agent_seg.py:1022-1065): NIfTI in, NIfTI out with the input
        volume's geometry (artefacts.py writes NIfTI-1 without SimpleITK); other names are saved as ``.npy``."""
        out_dir = self.config['testing'].get('output_dir', None)
        if not out_dir:
            return
        from . import artefacts
        os.makedirs(out_dir, exist_ok=True)
        root = self.config.get('dataset', {}).get('root_dir', '') or ''
        for name, lab in outputs.items():
            base = os.path.basename(str(name))
            vol = np.asarray(lab)
            vol = vol[0] if vol.ndim == 4 else vol
            if base.endswith(('.nii.gz', '.nii')):
                src = os.path.join(root, str(name))
                artefacts.save_array_as_nifty_volume(vol, os.path.join(out_dir, base), src if os.path.isfile(src) else None)
                continue
            for ext in ('.npy',):
                if base.endswith(ext):
                    base = base[:-len(ext)]
            np.save(os.path.join(out_dir, base + '.npy'), lab)

    def run(self):
        self.create_dataset()
        self.create_network()
        if self.stage == 'train':
            return self.train_valid()
        return self.infer()


def pixel_weights_from_pseudo_labels(logits_tgt, logits_src, image_weight=None):
    """Stage 3 of the FPL+ recipe on the device (data/get_pixel_weight.py:12-28 on the two
    Inferer outputs of one target volume): labels of both passes, agreement weight, count."""
    return fpl.agreement_weight(logits_tgt, logits_src, image_weight=image_weight)
