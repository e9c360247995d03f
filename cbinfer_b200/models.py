"""Random-init model builders for the BASELINE configs (the callers either side of the hot path).

* :func:`sceneLabelingBaseline` -- the 11-slot scene-labeling CNN whose topology is pinned by the
  reference's ``sceneLabeling/modelLoader.py:9-10,47,72-78`` (three KxK convs with ReLU, two
  2x2 max-pools, two trailing 1x1 convs); channel widths / 7x7 follow the authors' papers (the
  weight file ``models/modelBaseline.net`` is not shipped, so weights are random-init).
* :func:`sceneLabelingCBinfer` -- the CBinfer version following the ``experimentIdx`` recipes of
  ``sceneLabeling/modelLoader.py:41-87``.
* :func:`poseModel` -- OpenPose-style CPM (VGG-19 stem + T stages) with the layer table of
  ``poseDetection/openPose/PoseModel.py:34-68``.
"""
import copy

import torch
import torch.nn as nn

from . import CBConv2d, CBPoolMax2d, convert, convertPools, shareWorkspace


def sceneLabelingBaseline(seed=0):
    g = torch.random.get_rng_state()
    torch.manual_seed(seed)
    m = nn.Sequential(
        nn.Conv2d(3, 16, 7, padding=3), nn.ReLU(), nn.MaxPool2d(2, 2),
        nn.Conv2d(16, 64, 7, padding=3), nn.ReLU(), nn.MaxPool2d(2, 2),
        nn.Conv2d(64, 256, 7, padding=3), nn.ReLU(),
        nn.Conv2d(256, 64, 1), nn.ReLU(),
        nn.Conv2d(64, 8, 1),
    ).eval()
    torch.random.set_rng_state(g)
    return m


def enableCandidateDetection(m, fusePool=True, maskedConv=True):
    """B200 extension (no reference counterpart): inside every nn.Sequential, let each CB layer
    hand its change set to a directly following CB layer as detection *candidates*, so that layer
    thresholds only the pixels that were just rewritten instead of re-scanning its whole input.
    Where the neighbours allow it, one kernel also does a neighbour's part of the frame: a pool runs
    the next conv's detection and a conv on the tile path pools in its epilogue (``fusePool``), and
    two trailing masked 1x1 layers run in one launch (``maskedConv``).  The launching module reads
    the neighbour's state; the neighbour learns of the work from the marker it receives in the
    ('changeIndexes', x, marker) tuple (DetectionDone / FrameDone) and records it itself.
    Results are identical to the dense scan (tests/test_gpu_modules.py)."""
    import torch.nn as nn
    for seq in [mm for mm in m.modules() if type(mm) is nn.Sequential]:
        kids = list(seq.children())
        for a, b in zip(kids[:-1], kids[1:]):
            if type(b) is CBConv2d and not b.finegrained:
                if type(a) is CBConv2d and not a.finegrained:
                    a.propChangeIndexes = True
                    b.candidateDetect = True
                elif type(a) is CBPoolMax2d:
                    a.propPooledIndexes = True
                    b.candidateDetect = True
                    if fusePool:             # pooling + b's detection in one kernel
                        a._fusedNext = [b]
        if fusePool:
            # conv -> pool -> conv: a conv on the tile path also pools in its epilogue (and runs the
            # detection of the conv after the pool there), cb_conv_update_tiled_pool
            for a, p, b in zip(kids[:-2], kids[1:-1], kids[2:]):
                if type(a) is CBConv2d and type(p) is CBPoolMax2d and type(b) is CBConv2d \
                        and p._fusedNext and not a.finegrained:
                    a._fusedPool = [p]
        if maskedConv:
            # a 1x1 layer fed by a CB conv whose own index list nobody needs as an exact list (it is
            # last, or feeds another candidate-detecting conv) skips the compaction altogether
            for i, b in enumerate(kids):
                if type(b) is CBConv2d and tuple(b.kernel_size) == (1, 1) and b.candidateDetect \
                        and i > 0 and type(kids[i - 1]) is CBConv2d:
                    nxt = kids[i + 1] if i + 1 < len(kids) else None
                    if nxt is None or (type(nxt) is CBConv2d and nxt.candidateDetect) \
                            or (not b.propChangeIndexes and type(nxt) is not CBPoolMax2d):
                        b.maskedConv = True
        # two trailing masked 1x1 layers: one kernel runs detect + contraction of both (cb_tail_update)
        if maskedConv and len(kids) >= 2:
            b, c = kids[-2], kids[-1]
            if type(b) is CBConv2d and type(c) is CBConv2d and b.maskedConv and c.maskedConv \
                    and not c.propChangeIndexes:
                b._fusedTail = [c]
    return m


def sceneLabelingCBinfer(baseline, experimentIdx=6, threshold=1e-1, convertAll=True,
                         clonePoolOutput=True, candidateDetect=False):
    """CBinfer scene-labeling model sharing the baseline's parameters.

    experimentIdx follows sceneLabeling/modelLoader.py:8-16:
      <=3 : plain conversion;  4: + feedback loop;  5/6: + change-based pooling with index
      propagation;  7: fine-grained convolution.
    ``convertAll=True`` converts the two trailing 1x1 convs as well (BASELINE config 2: "all
    conv+maxpool converted"); ``False`` keeps them dense as modelLoader.py:65 does.
    """
    m = convert(copy.deepcopy(baseline), threshold=threshold)
    if not convertAll:
        kids = list(m.named_children())
        dense_tail = list(baseline.children())[8:11]
        m = nn.Sequential()
        for name, node in kids[:5]:
            m.add_module(name, node)
        for i, node in enumerate(dense_tail):
            m.add_module(str(8 + i), copy.deepcopy(node))
    convs = [mm for mm in m.modules() if type(mm) is CBConv2d]
    if experimentIdx >= 3:
        for c in convs:
            c.copyInput = False
    if experimentIdx in (4, 5, 6):
        for c in convs:
            c.feedbackLoop = True
    if experimentIdx in (5, 6):
        m = convertPools(m)
        for p in m.modules():
            if type(p) is CBPoolMax2d:
                p.cloneOutput = clonePoolOutput
    if experimentIdx == 7:
        for c in convs:
            c.finegrained = True
    if candidateDetect:
        enableCandidateDetection(m)
    return m.eval()


def calibrateThresholds(baseline, cbmodel, frame, factor=0.02):
    """Fixed per-layer thresholds for throughput runs (SURVEY section 8d): factor * (max - min) of
    the dense activation feeding each CB conv, measured on one frame."""
    feeds = {}
    hooks = []
    convs_dense = [mm for mm in baseline.modules() if type(mm) is nn.Conv2d]
    for i, c in enumerate(convs_dense):
        hooks.append(c.register_forward_hook(
            lambda mod, inp, out, i=i: feeds.__setitem__(i, float(inp[0].max() - inp[0].min()))))
    with torch.no_grad():
        baseline(frame)
    for h in hooks:
        h.remove()
    cbs = [mm for mm in cbmodel.modules() if type(mm) is CBConv2d]
    for i, c in enumerate(cbs):
        c.threshold = factor * feeds[i]
    return [c.threshold for c in cbs]


# ---- OpenPose-style CPM (poseDetection/openPose/PoseModel.py:34-68) ---------------------------

def _stage(cfg):
    layers = []
    for i, (cin, cout, k) in enumerate(cfg):
        layers.append(nn.Conv2d(cin, cout, k, padding=k // 2))
        if i != len(cfg) - 1:
            layers.append(nn.ReLU(inplace=True))
    return nn.Sequential(*layers)


class PoseModel(nn.Module):
    def __init__(self, T=6, seed=0):
        super(PoseModel, self).__init__()
        assert 1 <= T <= 6
        self.T = T
        g = torch.random.get_rng_state()
        torch.manual_seed(seed)
        vgg = [(3, 64), (64, 64), 'P', (64, 128), (128, 128), 'P', (128, 256), (256, 256),
               (256, 256), (256, 256), 'P', (256, 512), (512, 512), (512, 256), (256, 128)]
        layers = []
        for v in vgg:
            if v == 'P':
                layers.append(nn.MaxPool2d(2, 2))
            else:
                layers += [nn.Conv2d(v[0], v[1], 3, padding=1), nn.ReLU(inplace=True)]
        self.model0 = nn.Sequential(*layers)
        for br, cout in ((1, 38), (2, 19)):
            setattr(self, 'model1_%d' % br, _stage([(128, 128, 3), (128, 128, 3), (128, 128, 3),
                                                    (128, 512, 1), (512, cout, 1)]))
            for t in range(2, T + 1):
                setattr(self, 'model%d_%d' % (t, br),
                        _stage([(185, 128, 7)] + [(128, 128, 7)] * 4 + [(128, 128, 1), (128, cout, 1)]))
        torch.random.set_rng_state(g)
        self.eval()

    # The two branches of a stage are independent: with parallelBranches=True branch 2 runs on a
    # side CUDA stream (fork / join around every stage), also inside a captured CUDA graph.  At batch
    # 1 the model is launch-latency-bound (92 convs, ~3 dependent launches each), so overlapping the
    # branches hides a good part of it.  (poseModelCBinfer gives the branches separate stream-K
    # workspaces, which this needs.)
    parallelBranches = False

    def __getstate__(self):
        d = self.__dict__.copy()
        d['_side'] = None                      # CUDA streams are per process
        return d

    def forward(self, x):
        feat = self.model0(x)
        tmp = feat
        par = self.parallelBranches and x.is_cuda
        if par and getattr(self, '_side', None) is None:
            self._side = torch.cuda.Stream(x.device)
        for t in range(1, self.T + 1):
            if par:
                cur = torch.cuda.current_stream(x.device)
                self._side.wait_stream(cur)
                with torch.cuda.stream(self._side):
                    S = getattr(self, 'model%d_2' % t)(tmp)
                L = getattr(self, 'model%d_1' % t)(tmp)
                cur.wait_stream(self._side)
                S.record_stream(cur)
                tmp.record_stream(self._side)
            else:
                L = getattr(self, 'model%d_1' % t)(tmp)
                S = getattr(self, 'model%d_2' % t)(tmp)
            if t != self.T:
                tmp = torch.cat([L, S, feat], 1)
        return L, S


def poseModelCBinfer(pose, threshold=1e-1, feedbackLoop=True, pools=True):
    """Convert every nn.Sequential block of a PoseModel (poseDetection/modelConverter.py:85-86
    sets feedbackLoop on all CB layers)."""
    m = copy.deepcopy(pose)
    for name, child in list(m.named_children()):
        if type(child) is nn.Sequential:
            c = convert(child, threshold=threshold)
            if pools:
                c = convertPools(c)
            setattr(m, name, c)
    for mm in m.modules():
        if type(mm) is CBConv2d:
            mm.feedbackLoop = feedbackLoop
            mm.copyInput = False
    # one stream-K workspace per chain of layers that run in order: trunk + branch 1, and branch 2
    # (the branches of a stage may overlap, PoseModel.parallelBranches)
    chains = [nn.ModuleList(), nn.ModuleList()]
    for name, child in m.named_children():
        chains[1 if name.endswith('_2') else 0].append(child)
    for ch in chains:
        shareWorkspace(ch)
    return m.eval()


def getCBModuleList(m):
    """the CBConv2d layers of a (sub)model in forward order (poseDetection/modelConverter.py:76-83)"""
    return [mm for mm in m.modules() if type(mm) is CBConv2d]


def tuneHierarchical(modelTest, tuneModules, lossTolFirst=5e-5, lossTolDefault=2e-6):
    """Block-wise threshold search of the reference's pose experiment 11
    (poseDetection/modelConverter.py:107-168), generalised from T=2 to any number of stages:
    all thresholds start at 0; the trunk ``model0`` is tuned together with ``model1_1``; then, stage
    by stage, branch 1 is tuned, its thresholds are stashed and zeroed while branch 2 of the same
    stage is tuned (so the two branches do not mask each other's loss), and restored afterwards.

    ``tuneModules(cbModuleList, lossToleranceList)`` runs the greedy search on the given layers -
    normally a closure over :func:`cbinfer_b200.tuneThresholdParameters` with the user's sequences
    (exactly what the reference script does).  Returns {block name: thresholds}."""
    allMods = getCBModuleList(modelTest)
    for m in allMods:
        m.threshold = 0
    names = dict(modelTest.named_children())
    out = {}
    t = 1
    while 'model%d_1' % t in names:
        b1, b2 = names['model%d_1' % t], names.get('model%d_2' % t)
        mods1 = getCBModuleList(b1)
        if t == 1 and 'model0' in names:
            mods = getCBModuleList(names['model0']) + mods1
            tuneModules(mods, [lossTolFirst] + [lossTolDefault] * (len(mods) - 1))
            out['model0'] = [m.threshold for m in getCBModuleList(names['model0'])]
        else:
            tuneModules(mods1, [lossTolDefault] * len(mods1))
        stash = [m.threshold for m in mods1]
        out['model%d_1' % t] = stash
        if b2 is not None:
            for m in mods1:
                m.threshold = 0
            mods2 = getCBModuleList(b2)
            tuneModules(mods2, [lossTolDefault] * len(mods2))
            out['model%d_2' % t] = [m.threshold for m in mods2]
            for m, th in zip(mods1, stash):
                m.threshold = th
        t += 1
    return out
