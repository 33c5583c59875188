"""Evaluation side of the reference's datasets: ``pre_eval`` (per-image metric pre-results) and ``evaluate``
(dataset-level reduction) with the reference's signatures, result-dict keys and ``eval_results`` key names
(``tiseg/datasets/custom.py:219-435``, ``tiseg/datasets/conic.py:126-323``).

Ground truth comes either from files laid out like the reference's converted datasets (``*_sem.png`` read with
pillow, ``*_inst.npy``; ``custom.py:252-259``) or from arrays handed in at construction.  ``pre_eval`` batches
all predictions of one call that share a shape into ONE pass over the CUDA library (the reference loops over
images on the CPU); ``evaluate`` is host arithmetic on a handful of numbers per image.
"""
import os
import os.path as osp
from collections import OrderedDict

import numpy as np

from . import metrics as M
from . import ops
from . import _lib
from ._lib import is_torch


def _table(columns):
    """Plain-text table from an ordered mapping name -> list of cells."""
    cols = [[str(k)] + [("%.2f" % v if isinstance(v, (float, np.floating)) else str(v)) for v in vals]
            for k, vals in columns.items()]
    widths = [max(len(c) for c in col) for col in cols]
    rows = zip(*cols)
    return "\n".join(" | ".join(c.rjust(w) for c, w in zip(r, widths)) for r in rows)


def _log(msg, logger=None):
    if logger is None:
        print(msg)
    elif hasattr(logger, "info"):
        logger.info(msg)


def _host(a):
    """Result array -> numpy.  For a CUDA tensor the library context is synchronised first: errors only a kernel can
    detect (an instance id outside the supported range) are raised HERE instead of being read back as wrong numbers."""
    if is_torch(a):
        if a.is_cuda:
            _lib.get_ctx(a.device.index).synchronize()
        return a.cpu().numpy()
    return np.asarray(a)


class CustomDataset:
    """Nuclei dataset evaluation (binary instance metrics + semantic metrics): custom.py."""

    CLASSES = ('background', 'nuclei')

    def __init__(self, data_infos=None, sem_gts=None, inst_gts=None, names=None, classes=None,
                 img_dir=None, ann_dir=None, img_suffix='.tif', sem_suffix='_sem.png', inst_suffix='_inst.npy',
                 split=None):
        if classes is not None:
            self.CLASSES = tuple(classes)
        self.sem_suffix, self.inst_suffix, self.img_suffix = sem_suffix, inst_suffix, img_suffix
        self._sem_gts, self._inst_gts = sem_gts, inst_gts
        if data_infos is None and ann_dir is not None:
            data_infos = self.load_annotations(img_dir, img_suffix, ann_dir, sem_suffix, inst_suffix, split)
        if data_infos is None:
            n = len(inst_gts)
            names = list(names) if names is not None else ["%d" % i for i in range(n)]
            data_infos = [dict(file_name=nm + img_suffix, sem_file_name=nm + sem_suffix, inst_file_name=nm + inst_suffix)
                          for nm in names]
        self.data_infos = data_infos

    def __len__(self):
        return len(self.data_infos)

    @staticmethod
    def load_annotations(img_dir, img_suffix, ann_dir, sem_suffix, inst_suffix, split=None):
        """File listing of custom.py:180-217: names from the split file or from the *_sem.png files."""
        if split is not None:
            names = [ln.strip() for ln in open(split) if ln.strip()]
        else:
            names = sorted(f[:-len(sem_suffix)] for f in os.listdir(ann_dir) if f.endswith(sem_suffix))
        return [dict(file_name=osp.join(img_dir or "", nm + img_suffix), sem_file_name=osp.join(ann_dir, nm + sem_suffix),
                     inst_file_name=osp.join(ann_dir, nm + inst_suffix)) for nm in names]

    # ---- ground truth
    def prefetch(self, indices, workers=8):
        """Start reading the ground truth of ``indices`` in the background (``custom.py:252-259`` reads it
        synchronously inside ``pre_eval``, one image at a time, between two GPU calls).  A pool of threads decodes
        the ``*_sem.png`` / loads the ``*_inst.npy`` files — PNG inflate and ``np.load`` release the GIL — so that
        by the time ``pre_eval`` asks for an index its arrays are in memory.  Call it for batch k+1 before running
        the model on batch k."""
        if self._inst_gts is not None:
            return
        import concurrent.futures
        if getattr(self, "_pool", None) is None:
            self._pool = concurrent.futures.ThreadPoolExecutor(max_workers=int(workers))
            self._pending = {}
        for i in indices:
            if i not in self._pending:
                self._pending[i] = self._pool.submit(self._read_gt, i)

    def _read_gt(self, index):
        from PIL import Image
        info = self.data_infos[index]
        sem_gt = np.array(Image.open(info['sem_file_name']))          # mmcv.imread(flag='unchanged', backend='pillow')
        inst_gt = np.load(info['inst_file_name'])
        return sem_gt, inst_gt

    def _load_gt(self, index):
        if self._inst_gts is not None:
            return self._sem_gts[index], self._inst_gts[index]
        pending = getattr(self, "_pending", None)
        if pending and index in pending:
            return pending.pop(index).result()
        from PIL import Image
        info = self.data_infos[index]
        sem_gt = np.array(Image.open(info['sem_file_name']))          # mmcv.imread(flag='unchanged', backend='pillow')
        inst_gt = np.load(info['inst_file_name'])
        return sem_gt, inst_gt

    def _gather(self, preds, indices):
        if not isinstance(indices, list):
            indices = [indices]
        if not isinstance(preds, list):
            preds = [preds]
        sem_gt, inst_gt = zip(*[self._load_gt(i) for i in indices])
        return preds, indices, sem_gt, inst_gt

    @staticmethod
    def _stack(arrs, dtype):
        """Same-shaped per-image arrays -> one batch (CUDA tensors stay on the device)."""
        if is_torch(arrs[0]):
            import torch
            if dtype == np.uint16:
                # stacked as int16 views (the same bits): torch implements few operators for uint16
                return torch.stack([a.view(torch.int16) for a in arrs]).view(torch.uint16)
            tdt = {np.uint8: torch.uint8, np.int32: torch.int32}[dtype]
            return torch.stack([a for a in arrs]).to(tdt)
        return np.stack([np.asarray(a) for a in arrs]).astype(dtype, copy=False)

    @staticmethod
    def _inst_dtype(arrs):
        """Batch dtype of a group of ground-truth instance maps: uint16 when every map of the group is uint16 (numpy or
        torch; the kernels read it as it is, at half the bytes of int32), int32 otherwise."""
        return np.uint16 if all(str(getattr(a, "dtype", "")) in ("uint16", "torch.uint16") for a in arrs) else np.int32

    def _groups(self, preds):
        by_shape = OrderedDict()
        for k, p in enumerate(preds):
            by_shape.setdefault(tuple(p['inst_pred'].shape), []).append(k)
        return by_shape.values()

    def pre_eval(self, preds, indices, show=False, show_folder=None):
        """custom.py:219-305.  preds: list of {'sem_pred', 'inst_pred'}; returns one dict per image with
        ``name``, ``bin_aji_pre_eval_res``, ``bin_pq_pre_eval_res``, ``sem_pre_eval_res``."""
        if show:
            raise NotImplementedError("drawing (show=True) is outside the rebuilt path")
        preds, indices, sem_gts, inst_gts = self._gather(preds, indices)
        out = [None] * len(preds)
        C = len(self.CLASSES)
        for ks in self._groups(preds):
            sem_p = self._stack([preds[k]['sem_pred'] for k in ks], np.uint8)
            inst_p = self._stack([preds[k]['inst_pred'] for k in ks], np.int32)
            sem_g = self._stack([sem_gts[k] for k in ks], np.uint8)        # CUDA-resident ground truth stays resident
            inst_g = self._stack([inst_gts[k] for k in ks], self._inst_dtype([inst_gts[k] for k in ks]))
            sem_res = M.pre_eval_all_semantic_metric(sem_p, sem_g, C)
            # re_instance + measure.label of both maps happen inside the pair kernel (custom.py:272-277)
            aji, pq = ops.pair_metrics_bin(inst_p, inst_g)
            aji, pq = _host(aji), _host(pq)
            for j, k in enumerate(ks):
                info = self.data_infos[indices[k]]
                data_id = osp.basename(info['sem_file_name']).replace(self.sem_suffix, '')
                out[k] = dict(
                    name=data_id,
                    bin_aji_pre_eval_res=(np.float64(aji[j, 0]), np.float64(aji[j, 1])),
                    bin_pq_pre_eval_res=(int(pq[j, 0]), int(pq[j, 1]), int(pq[j, 2]), np.float64(pq[j, 3])),
                    sem_pre_eval_res=sem_res[j])
        return out

    # ---- batched records (no per-image Python): what a multi-GPU sweep accumulates and exchanges
    def _gt_batch(self, indices):
        """ground truth of `indices` as two stacked arrays; a contiguous range of GT held as one stacked tensor / array
        is a slice, not a copy"""
        sem, inst = self._sem_gts, self._inst_gts
        contiguous = len(indices) > 0 and list(indices) == list(range(indices[0], indices[0] + len(indices)))
        if inst is not None and not isinstance(inst, (list, tuple)) and contiguous:
            return sem[indices[0]:indices[0] + len(indices)], inst[indices[0]:indices[0] + len(indices)]
        sg, ig = zip(*[self._load_gt(i) for i in indices])
        return self._stack(list(sg), np.uint8), self._stack(list(ig), self._inst_dtype(ig))

    def pre_eval_records(self, sem_pred, inst_pred, indices, check=True):
        """``pre_eval`` for a whole batch ``[n, H, W]`` without a Python loop over the images: returns ONE float64 array
        / tensor ``[n, R]`` in the layout of ``parallel.pack_results`` (bin aji 2, bin pq 4, sem 6 x (C-1), and for
        multi-class datasets aji 2 x (C-1), pq 4 x (C-1)); ``parallel.unpack_results`` turns rows back into the
        per-image dictionaries ``evaluate`` takes.  Values are what ``pre_eval`` would have put in the dictionaries.
        ``check``: synchronise the library context before returning device results, so that errors only a kernel can
        detect (an instance id outside the supported range) are raised here, once per batch; pass False to keep the
        batch asynchronous and call ``tiseg_b200._lib.get_ctx(device).synchronize()`` yourself before reading."""
        import torch
        C = len(self.CLASSES)
        sem_g, inst_g = self._gt_batch(list(indices))
        multi = isinstance(self, CoNICDataset)
        counts, _ = ops.sem_counts(sem_pred, sem_g, C)
        if multi:
            r = ops.pair_metrics_multiclass(inst_pred, sem_pred, inst_g, sem_g, C)
            baji, bpq, caji, cpq = r['bin_aji'], r['bin_pq'], r['aji'], r['pq']
        else:
            baji, bpq = ops.pair_metrics_bin(inst_pred, inst_g)
        t = (lambda a: a if is_torch(a) else torch.from_numpy(np.asarray(a)))
        counts = t(counts).float()                                      # the reference keeps these in float32
        tp, fp, fn, pr, gt = (counts[:, k] for k in range(5))
        tn = pr.sum(1, keepdim=True) - (tp + fp + fn)                   # sem_metrics.py:43
        f32 = lambda a: a.float().double()
        parts = [t(baji), t(bpq)] + [x[:, 1:].double() for x in (tp, tn, fp, fn, pr, gt)]
        if multi:
            ca, cq = t(caji), t(cpq)
            parts += [f32(ca[:, 1:, k]) for k in range(2)] + [f32(cq[:, 1:, k]) for k in range(4)]
        rec = torch.cat(parts, dim=1)
        if check and rec.is_cuda:
            _lib.get_ctx(rec.device.index).synchronize()
        return rec

    @staticmethod
    def _columns(results):
        cols = {}
        for r in results:
            for k, v in r.items():
                cols.setdefault(k, []).append(v)
        return cols

    def evaluate(self, results, logger=None, **kwargs):
        """custom.py:307-435 -> (eval_results, storage_results)."""
        ret, img = self._columns(results), {}
        names = ret.pop('name')
        sem = ret.pop('sem_pre_eval_res')
        ret.update(M.pre_eval_to_sem_metrics(sem, metrics=['Dice', 'Precision', 'Recall']))
        img.update(M.pre_eval_to_imw_sem_metrics(sem, metrics=['Dice', 'Precision', 'Recall']))
        baji = ret.pop('bin_aji_pre_eval_res')
        ret.update(M.pre_eval_to_aji(baji))
        ret.update({'b' + k: v for k, v in M.pre_eval_to_bin_aji(baji).items()})
        img.update(M.pre_eval_to_imw_aji(baji))
        bpq = ret.pop('bin_pq_pre_eval_res')
        ret.update(M.pre_eval_to_pq(bpq))
        ret.update({'b' + k: v for k, v in M.pre_eval_to_bin_pq(bpq).items()})
        ret.update(M.pre_eval_to_inst_dice(bpq))
        img.update(M.pre_eval_to_imw_pq(bpq))
        img.update(M.pre_eval_to_imw_inst_dice(bpq))

        names = list(names) + ['Average']
        for key in img:
            v = np.asarray(img[key])
            if v.ndim == 2:
                v = v[:, 0]
            # custom.py:367-370: the list round trip turns the float32 semantic columns into float64
            lst = v.tolist()
            lst.append(np.nanmean(v))
            img[key] = np.array(lst)

        vital = ['Dice', 'Precision', 'Recall', 'Aji', 'DQ', 'SQ', 'PQ', 'InstDice']
        mean_metrics = OrderedDict(('imw' + k, img[k][-1]) for k in vital)
        overall = OrderedDict(('m' + k, ret[k]) for k in vital)
        for k in ['bAji', 'bDQ', 'bSQ', 'bPQ']:
            overall[k] = ret[k]

        sample = OrderedDict(name=names)
        sample.update((k, np.round(np.asarray(v) * 100, 2)) for k, v in img.items())
        _log('Per samples:\n' + _table(sample), logger)
        mean_metrics = OrderedDict((k, np.round(np.mean(v) * 100, 2)) for k, v in mean_metrics.items())
        overall = OrderedDict((k, np.round(np.mean(v) * 100, 2)) for k, v in overall.items())
        _log('Mean Total:\n' + _table(OrderedDict((k, [v]) for k, v in mean_metrics.items())), logger)
        _log('Overall Total:\n' + _table(OrderedDict((k, [v]) for k, v in overall.items())), logger)

        storage_results = {'mean_metrics': mean_metrics, 'overall_metrics': overall}
        eval_results = {}
        eval_results.update(mean_metrics)
        eval_results.update(overall)
        return eval_results, storage_results


class MoNuSegDataset(CustomDataset):
    CLASSES = ('background', 'nuclei')


class GlasDataset(CustomDataset):       # glas.py: '.png' images
    CLASSES = ('background', 'nuclei')

    def __init__(self, *args, **kwargs):
        kwargs.setdefault('img_suffix', '.png')
        super().__init__(*args, **kwargs)


class MoNuSegDatasetDebug(CustomDataset):
    """monuseg_debug.py: the predictions also carry the three-class maps ``tc_pred`` / ``tc_gt`` and the evaluation
    adds the boundary class's Dice / Precision / Recall (``BoundDice`` ...)."""
    CLASSES = ('background', 'nuclei')

    def pre_eval(self, preds, indices, show=False, show_folder=None):
        out = super().pre_eval(preds, indices, show, show_folder)
        if not isinstance(preds, list):
            preds = [preds]
        C = len(self.CLASSES) + 1
        for ks in self._groups(preds):
            tc_p = self._stack([preds[k]['tc_pred'] for k in ks], np.uint8)
            tc_g = self._stack([preds[k]['tc_gt'] for k in ks], np.uint8)
            res = M.pre_eval_all_semantic_metric(tc_p, tc_g, C)            # monuseg_debug.py:85
            for j, k in enumerate(ks):
                out[k]['bound_sem_pre_eval_res'] = res[j]
        return out

    def evaluate(self, results, logger=None, **kwargs):
        bound = [r['bound_sem_pre_eval_res'] for r in results]
        rest = [{k: v for k, v in r.items() if k != 'bound_sem_pre_eval_res'} for r in results]
        eval_results, storage = super().evaluate(rest, logger=logger, **kwargs)
        bm = M.pre_eval_to_sem_metrics(bound, metrics=['Dice', 'Precision', 'Recall'])      # :133-135: the last class
        extra = OrderedDict(('Bound' + k, np.round(np.mean(v[-1]) * 100, 2)) for k, v in bm.items())
        storage['overall_metrics'].update(extra)
        eval_results.update(extra)
        return eval_results, storage


class CPM17Dataset(CustomDataset):
    CLASSES = ('background', 'nuclei')


class CoNSePDataset(CustomDataset):
    CLASSES = ('background', 'nuclei')


class CoNICDataset(CustomDataset):
    """Multi-class nuclei evaluation: conic.py."""

    CLASSES = ('background', 'neutrophil', 'epithelial', 'lymphocyte', 'plasma', 'eosinophil', 'connective')

    def pre_eval(self, preds, indices, show=False, show_folder='.nuclei_show'):
        """conic.py:126-198: adds the per-class ``aji_pre_eval_res`` / ``pq_pre_eval_res``."""
        if show:
            raise NotImplementedError("drawing (show=True) is outside the rebuilt path")
        preds, indices, sem_gts, inst_gts = self._gather(preds, indices)
        out = [None] * len(preds)
        C = len(self.CLASSES)
        for ks in self._groups(preds):
            sem_p = self._stack([preds[k]['sem_pred'] for k in ks], np.uint8)
            inst_p = self._stack([preds[k]['inst_pred'] for k in ks], np.int32)
            sem_g = self._stack([sem_gts[k] for k in ks], np.uint8)        # CUDA-resident ground truth stays resident
            inst_g = self._stack([inst_gts[k] for k in ks], self._inst_dtype([inst_gts[k] for k in ks]))
            sem_res = M.pre_eval_all_semantic_metric(sem_p, sem_g, C)
            r = ops.pair_metrics_multiclass(inst_p, sem_p, inst_g, sem_g, C)
            aji, pq = _host(r['aji']).astype(np.float32), _host(r['pq']).astype(np.float32)
            baji, bpq = _host(r['bin_aji']), _host(r['bin_pq'])
            for j, k in enumerate(ks):
                out[k] = dict(
                    bin_aji_pre_eval_res=(np.float64(baji[j, 0]), np.float64(baji[j, 1])),
                    aji_pre_eval_res=(aji[j, 1:, 0], aji[j, 1:, 1]),
                    bin_pq_pre_eval_res=(int(bpq[j, 0]), int(bpq[j, 1]), int(bpq[j, 2]), np.float64(bpq[j, 3])),
                    pq_pre_eval_res=tuple(pq[j, 1:, q] for q in range(4)),
                    sem_pre_eval_res=sem_res[j])
        return out

    def evaluate(self, results, logger=None, **kwargs):
        """conic.py:200-323 -> (eval_results, storage_results) incl. the per-class ``Metric.class`` entries."""
        ret, img = self._columns(results), {}
        ret.pop('name', None)
        sem = ret.pop('sem_pre_eval_res')
        ret.update(M.pre_eval_to_sem_metrics(sem, metrics=['Dice', 'Precision', 'Recall']))
        img.update(M.pre_eval_to_imw_sem_metrics(sem, metrics=['Dice', 'Precision', 'Recall']))
        aji, baji = ret.pop('aji_pre_eval_res'), ret.pop('bin_aji_pre_eval_res')
        ret.update(M.pre_eval_to_aji(aji))
        ret.update({'b' + k: v for k, v in M.pre_eval_to_bin_aji(baji).items()})
        img.update(M.pre_eval_to_imw_aji(baji))
        pq, bpq = ret.pop('pq_pre_eval_res'), ret.pop('bin_pq_pre_eval_res')
        ret.update(M.pre_eval_to_pq(pq))
        ret.update({'b' + k: v for k, v in M.pre_eval_to_bin_pq(bpq).items()})
        img.update(M.pre_eval_to_imw_pq(bpq))

        vital = ['Dice', 'Precision', 'Recall', 'Aji', 'DQ', 'SQ', 'PQ']
        mean_metrics, overall, per_class = OrderedDict(), OrderedDict(), OrderedDict()
        for k in vital:
            mean_metrics['imw' + k] = np.nanmean(img[k])
            overall['m' + k] = np.nanmean(ret[k])
            v = np.asarray(ret[k], dtype=np.float64).ravel()
            per_class[k] = np.round(np.append(v, np.nanmean(v)) * 100, 2)
        for k in ['bAji', 'bDQ', 'bSQ', 'bPQ']:
            overall[k] = ret[k]
        classes = list(self.CLASSES[1:]) + ['average']
        tab = OrderedDict(classes=classes)
        tab.update(per_class)
        _log('Per classes:\n' + _table(tab), logger)
        mean_metrics = OrderedDict((k, np.round(np.mean(v) * 100, 2)) for k, v in mean_metrics.items())
        overall = OrderedDict((k, np.round(np.mean(v) * 100, 2)) for k, v in overall.items())
        _log('Mean Total:\n' + _table(OrderedDict((k, [v]) for k, v in mean_metrics.items())), logger)
        _log('Overall Total:\n' + _table(OrderedDict((k, [v]) for k, v in overall.items())), logger)
        storage_results = {'mean_metrics': mean_metrics, 'overall_metrics': overall}
        eval_results = {}
        eval_results.update(overall)
        eval_results.update(mean_metrics)
        for key, value in per_class.items():
            eval_results.update({key + '.' + str(name): f'{value[idx]:.3f}' for idx, name in enumerate(classes)})
        return eval_results, storage_results
