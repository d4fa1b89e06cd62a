"""oracle/ref_layers.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE (dev container only).

Runs the reference's OWN Python layers in place: the ``ClassDef`` nodes of SoftmaxLayer,
BalancedSeedLossLayer, ConstrainLossLayer and AnnotationLayer are pulled out of
/root/reference/pylayers/pylayers/pylayers.py with ``ast`` (the module itself cannot be imported: it
needs caffe, theano and cPickle at import time; nothing is copied) and executed against
``oracle/theano_shim`` (the Theano stand-in) and a minimal Blob/Layer stand-in for pycaffe.  The outputs
are what pins ``oracle/loss_oracle.py`` and ``oracle/annot_oracle.py``: tests/golden/make_golden.py
freezes them in tests/golden/layers_ref.npz and layers_ref_sweep.npz, which tests/test_oracle_golden.py
compares against.
"""
import ast
import os
import types

import numpy as np

from . import theano_shim

REF_FILE = "/root/reference/pylayers/pylayers/pylayers.py"
WANTED = ("SoftmaxLayer", "BalancedSeedLossLayer", "ConstrainLossLayer", "AnnotationLayer")
_NS = None


def available():
    return os.path.exists(REF_FILE)


class Blob(object):
    def __init__(self, data=None):
        self.data = np.zeros((1,), np.float32) if data is None else np.array(data, np.float32)
        self.diff = np.zeros_like(self.data)

    def reshape(self, *shape):
        if tuple(shape) != self.data.shape:
            self.data = np.zeros(shape, np.float32)
            self.diff = np.zeros(shape, np.float32)


def namespace():
    """The reference's layer classes, defined by executing their own source in place."""
    global _NS
    if _NS is None:
        with open(REF_FILE) as fh:
            tree = ast.parse(fh.read())
        keep = [n for n in tree.body
                if (isinstance(n, ast.ClassDef) and n.name in WANTED) or
                (isinstance(n, ast.Assign) and all(isinstance(t, ast.Name) for t in n.targets))]
        theano, T = theano_shim.install()
        caffe = types.ModuleType("caffe")
        caffe.Layer = type("Layer", (object,), {"param_str": ""})
        ns = {"np": np, "caffe": caffe, "theano": theano, "T": T, "osp": os.path}
        exec(compile(ast.Module(body=keep, type_ignores=[]), REF_FILE, "exec"), ns)
        _NS = ns
    return _NS


def _run(name, bottoms, top_diff=None, n_top=1, dtype="float32"):
    """setup -> reshape -> forward -> backward of the reference layer `name` on numpy inputs."""
    import torch
    theano_shim.set_dtype(torch.float64 if dtype == "float64" else torch.float32)
    try:
        layer = namespace()[name]()
        bottom = [Blob(b) for b in bottoms]
        if dtype == "float64":   # keep the inputs exact: Blob() rounds to float32 like Caffe does
            for bl, b in zip(bottom, bottoms):
                bl.data = np.array(b, np.float64)
                bl.diff = np.zeros_like(bl.data)
        top = [Blob() for _ in range(n_top)]
        if dtype == "float64":
            for t in top:
                t.data = t.data.astype(np.float64)
                t.diff = t.diff.astype(np.float64)
        layer.setup(bottom, top)
        layer.reshape(bottom, top)
        if dtype == "float64":
            for t in top:
                t.data = t.data.astype(np.float64)
                t.diff = t.diff.astype(np.float64)
        layer.forward(bottom, top)
        if top_diff is not None:
            top[0].diff[...] = top_diff
        layer.backward(top, [True] * len(bottom), bottom)
        return [np.array(t.data) for t in top], [np.array(b.diff) for b in bottom]
    finally:
        theano_shim.set_dtype(torch.float32)


def softmax_layer(preds, top_diff, dtype="float32"):
    """(probs, d preds): pylayers.py:23-51."""
    tops, diffs = _run("SoftmaxLayer", [preds], top_diff, dtype=dtype)
    return tops[0], diffs[0]


def balanced_seed_loss_layer(probs, labels, dtype="float32"):
    """(loss, d probs): pylayers.py:120-152."""
    tops, diffs = _run("BalancedSeedLossLayer", [probs, labels], dtype=dtype)
    return tops[0].reshape(-1)[0], diffs[0]


def constrain_loss_layer(probs, log_smooth, dtype="float32"):
    """(loss, d probs, d log_smooth): pylayers.py:154-180."""
    tops, diffs = _run("ConstrainLossLayer", [probs, log_smooth], dtype=dtype)
    return tops[0].reshape(-1)[0], diffs[0], diffs[1]


def annotation_layer_forward(data_file, image_ids, images, is_mirror, seed=None):
    """The reference's own AnnotationLayer.forward (pylayers.py:369-387) on an in-memory cue dictionary
    (setup() is skipped: it only parses param_str and unpickles the cue file, :348-362)."""
    layer = namespace()["AnnotationLayer"]()
    layer.data_file = data_file
    layer.is_mirror = is_mirror
    bottom = [Blob(np.asarray(image_ids, np.float32).reshape(-1)), Blob(images)]
    top = [Blob(), Blob(), Blob()]
    layer.reshape(bottom, top)
    if seed is not None:
        np.random.seed(seed)
    layer.forward(bottom, top)
    return top[0].data, top[1].data, top[2].data
