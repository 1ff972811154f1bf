"""Drop-in ``Inferer`` (reference: PyMIC/pymic/net_run_dsbn/infer_func.py:6-222): sliding-window
inference with overlap averaging and 4-flip test-time augmentation, same config keys
(``sliding_window_enable/size/stride``, ``tta_mode``, ``class_num``) and the same
``run(model, image, domain_label)`` call.

B200 re-design: all windows of a pass are stacked into ONE batched network call (exact for a
network in eval mode, where BatchNorm uses running statistics), window results are scattered
into the volume by a fused accumulate kernel and normalised by the visit count on the device;
the un-flip of TTA passes is folded into the accumulate kernel.  The reference's probe forward
on a ones tensor (infer_func.py:92-93) is not issued: it only counts outputs.
"""
import ctypes

import torch

from .ops import call, ptr, stream_ptr


def _bn_in_eval(model):
    for m in model.modules():
        if isinstance(m, torch.nn.modules.batchnorm._BatchNorm) and m.training:
            return False
    return True


class Inferer(object):
    def __init__(self, config):
        self.config = config
        self.max_batch = config.get('window_batch', 8)
        self._side = None

    # window enumeration: infer_func.py:55-85 (w outer, h, d inner; last window clamped)
    def _windows(self, img_shape):
        win = [x for x in self.config['sliding_window_size']]
        stride = [x for x in self.config['sliding_window_stride']]
        if len(img_shape) != 3:
            raise ValueError("Inference using sliding window only supports 3D images here")
        for d in range(3):
            if win[d] is None or win[d] > img_shape[d]:
                win[d] = img_shape[d]
            if stride[d] is None or stride[d] > win[d]:
                stride[d] = win[d]
        if all(win[d] >= img_shape[d] for d in range(3)):
            return None, win
        starts = []
        for w in range(0, img_shape[2], stride[2]):
            w0 = min(w, img_shape[2] - win[2])
            for h in range(0, img_shape[1], stride[1]):
                h0 = min(h, img_shape[1] - win[1])
                for d in range(0, img_shape[0], stride[0]):
                    starts.append((min(d, img_shape[0] - win[0]), h0, w0))
        return starts, win

    def _model(self, x, domain_label, lane=None, repeats=1):
        """Returns a list of ``repeats`` outputs (MC-dropout passes of the same input share their dropout-free
        encoder prefix through ``forward_mc`` when the model offers it)."""
        if repeats > 1:
            if hasattr(self.model, "forward_mc"):
                return self.model.forward_mc(x, domain_label, repeats, graph_lane=0 if lane is None else lane)
            return [self._model(x, domain_label, lane)[0] for _ in range(repeats)]
        if lane is None:
            out = self.model(x, domain_label=domain_label)
        else:
            out = self.model(x, domain_label=domain_label, graph_lane=lane)
        if isinstance(out, (tuple, list)):
            out = out[0]
        return [out]

    def _two_lanes(self, model):
        """The fplplus_b200 network accepts ``graph_lane``: two half-batches of windows can then run concurrently
        on two streams (tensor-pipe-bound convolutions of one under the HBM-bound BatchNorm kernels of the other)."""
        return self.config.get('window_two_streams', True) and hasattr(model, "_forward_graphed") and model.cuda_graphs

    def _infer(self, image, domain_label, results, scale, flip_h, flip_w):
        """results[k] += scale * unflip(sliding_window(model, image)) for each of the len(results) MC passes."""
        K = len(results)
        b, _cin, vd, vh, vw = image.shape
        class_num = self.config['class_num']
        st = stream_ptr()
        starts = None
        if self.config.get('sliding_window_enable', False):
            starts, win = self._windows([vd, vh, vw])
        if starts is None:
            for k, out in enumerate(self._model(image, domain_label, None, K)):
                out = out.float().contiguous()
                call("fpl_window_accumulate", ptr(out), ptr(results[k]), None, b, out.shape[1], vd, vh, vw, 0, 0, 0,
                     vd, vh, vw, flip_h, flip_w, scale, st)
            return
        accs = [torch.zeros((b, class_num, vd, vh, vw), dtype=torch.float32, device=image.device) for _ in range(K)]
        acc = accs[0]
        cnt = torch.zeros_like(acc)
        batched = _bn_in_eval(self.model)
        group = max(1, self.max_batch // b) if batched else 1
        two = batched and self._two_lanes(self.model) and len(starts) >= 2
        main = torch.cuda.current_stream()
        if two:
            if self._side is None:
                self._side = torch.cuda.Stream()
            # each lane accumulates into its own volume (windows of the two lanes may overlap): deterministic sums
            accs1, cnt1 = [torch.zeros_like(acc) for _ in range(K)], torch.zeros_like(cnt)
            # stale weight images are re-staged HERE, on the main stream, before the side stream forks: lane 0 would
            # otherwise stage them lazily after the fork and lane 1 could read half-written images
            prepare = getattr(self.model, "prepare", None)
            if prepare is not None:
                prepare((b,) + tuple(image.shape[1:2]) + tuple(win), grad=False)
            self._side.wait_stream(main)
            group = max(1, group // 2)
        lane = 0
        for g0 in range(0, len(starts), group):
            chunk = starts[g0:g0 + group]
            stream = self._side if (two and lane == 1) else main
            with torch.cuda.stream(stream):
                patches = [image[:, :, d0:d0 + win[0], h0:h0 + win[1], w0:w0 + win[2]] for d0, h0, w0 in chunk]
                x = torch.cat(patches, 0).contiguous() if len(patches) > 1 else patches[0].contiguous()
                dl = domain_label if len(chunk) == 1 else domain_label.repeat(len(chunk))
                outs = self._model(x, dl, lane if two else None, K)
                sp = ctypes.c_void_p(stream.cuda_stream)
                as_, c_ = (accs1, cnt1) if (two and lane == 1) else (accs, cnt)
                for k, out in enumerate(outs):
                    out = out.float().contiguous()
                    for j, (d0, h0, w0) in enumerate(chunk):
                        # the visit count is the same for every pass: accumulated with pass 0 only
                        call("fpl_window_accumulate", ptr(out[j * b:(j + 1) * b]), ptr(as_[k]), ptr(c_) if k == 0 else None, b,
                             class_num, vd, vh, vw, d0, h0, w0, win[0], win[1], win[2], 0, 0, 1.0, sp)
            if two:
                lane ^= 1
        if two:
            main.wait_stream(self._side)
            for k in range(K):
                accs[k].add_(accs1[k])
            cnt.add_(cnt1)
        for k in range(K):
            call("fpl_window_normalize", ptr(accs[k]), ptr(cnt), 1.0, acc.numel(), st)
            call("fpl_window_accumulate", ptr(accs[k]), ptr(results[k]), None, b, class_num, vd, vh, vw, 0, 0, 0, vd, vh, vw,
                 flip_h, flip_w, scale, st)

    def run(self, model, image, domain_label, mc_passes=1):
        """Logits [B,class_num,D,H,W] on ``image.device`` (infer_func.py:188-222).  ``mc_passes`` = K > 1: the K
        MC-dropout passes of agent_seg.py:897-911 over the same volume in one sweep (a list of K logits volumes)."""
        self.model = model
        if mc_passes > 1 and hasattr(model, "kMaxMcRepeats") and mc_passes > model.kMaxMcRepeats:
            raise ValueError("mc_passes = %d exceeds %d" % (mc_passes, model.kMaxMcRepeats))
        tta_mode = self.config.get('tta_mode', 0)
        if tta_mode not in (0, 1):
            raise ValueError("Undefined tta_mode {0:}".format(tta_mode))
        image = image.float()
        b, _c, vd, vh, vw = image.shape
        class_num = self.config['class_num']
        results = [torch.zeros((b, class_num, vd, vh, vw), dtype=torch.float32, device=image.device)
                   for _ in range(max(1, int(mc_passes)))]
        if tta_mode == 0:
            self._infer(image, domain_label, results, 1.0, 0, 0)
        else:
            self._infer(image, domain_label, results, 0.25, 0, 0)
            self._infer(torch.flip(image, [-2]), domain_label, results, 0.25, 1, 0)
            self._infer(torch.flip(image, [-1]), domain_label, results, 0.25, 0, 1)
            self._infer(torch.flip(image, [-2, -1]), domain_label, results, 0.25, 1, 1)
        return results if mc_passes > 1 else results[0]
