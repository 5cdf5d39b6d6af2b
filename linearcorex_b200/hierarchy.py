"""Hierarchical Linear CorEx: the layer-stacking loop of the reference CLI (vis_corex.py:529-545).

Layer 0 fits X (with the missing-value marker); layer k > 0 fits `transform()` of layer k-1 (no marker);
a final one-unit layer is appended when the last width is not 1 (vis_corex.py:489-491).  Unlike the CLI
the intermediate representations never leave the GPU: layer k's Y stays a row-sharded CUDA tensor and is
handed to layer k+1's `fit` directly (SURVEY.md section 8(f) item 1).
"""
from .corex import Corex


def fit_layers(x, layers, missing_values=None, gaussianize='standard', discourage_overlap=True, max_iter=10000,
               tol=1e-5, seed=None, verbose=False, sample_weight=None, **corex_kwargs):
    """Fit a stack of Corex layers.  Returns the list of fitted models (layer 0 first).

    `seed` is passed to every layer (the reference CLI never seeds, vis_corex.py:535-545); `corex_kwargs`
    forwards the B200 extensions (`precision`, `exact_trials`, `comm`, `device`, ...).  `sample_weight` (one
    per row of x) is passed to every layer's fit: the rows of layer k's input are the rows of x."""
    layers = [int(v) for v in layers]
    if layers[-1] != 1:
        layers.append(1)  # last layer has one unit so the graph is fully connected
    models, x_prev = [], x
    for depth, width in enumerate(layers):
        kw = dict(n_hidden=width, verbose=verbose, gaussianize=gaussianize, discourage_overlap=discourage_overlap,
                  max_iter=max_iter, tol=tol, seed=seed, **corex_kwargs)
        if depth == 0:
            kw["missing_values"] = missing_values
        else:
            x_prev = models[-1].transform(x_prev, return_device=True)
        models.append(Corex(**kw).fit(x_prev, sample_weight=sample_weight))
    return models


def transform_layers(models, x):
    """Representations of x at every layer (host arrays), like chaining `transform` in the CLI."""
    out, cur = [], x
    for mdl in models:
        cur = mdl.transform(cur, return_device=True)
        out.append(cur.cpu().numpy().copy())
    return out
