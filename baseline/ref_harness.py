"""The UNMODIFIED reference (yjxiong/action-detection) as bench.py's `--impl reference` arm and as the CPU baseline.

The reference is run from a checkout of it named by the environment variable SSNB_REFERENCE_DIR, imported where it is:
nothing is copied into this repository.  Without that variable bench.py falls back to the oracle port.  No reference file
is edited: four monkey-patches are applied from outside (SURVEY.md section 8c):
  1. yaml.load gets a default Loader           (model_zoo/bninception/pytorch_load.py:13 predates PyYAML 6)
  2. torch.utils.model_zoo.load_url -> None    (pytorch_load.py:35 downloads pretrained weights; no network)
  3. BNInception.load_state_dict -> no-op      (during construction only; seeded synthetic weights are loaded afterwards)
  4. torch.Tensor.cuda -> identity             (ops/ssn_ops.py:113-120,192,213 hard-code .cuda(); this arm runs on the CPU)
This module is benchmark infrastructure: the product package never imports it.
"""
import contextlib
import io
import os
import sys
import warnings

REF = os.path.abspath(os.environ["SSNB_REFERENCE_DIR"]) if os.environ.get("SSNB_REFERENCE_DIR") else None


def available():
    return REF is not None and os.path.exists(os.path.join(REF, "ssn_models.py"))


_mods = None


def import_reference():
    """-> (ssn_models, ops.ssn_ops) of the reference checkout, patches 1-4 applied"""
    global _mods
    if _mods is not None:
        return _mods
    if not available():
        raise ImportError("no reference checkout: set SSNB_REFERENCE_DIR to the root of yjxiong/action-detection")
    import torch
    import yaml
    _orig = yaml.load
    yaml.load = lambda s, Loader=yaml.SafeLoader: _orig(s, Loader=Loader)
    import torch.utils.model_zoo as mz
    mz.load_url = lambda *a, **k: None
    torch.Tensor.cuda = lambda self, *a, **k: self
    warnings.filterwarnings("ignore")
    # the reference's top-level module names (ssn_models, ops, model_zoo, transforms) are also the names of this repo's
    # drop-in package: the reference arm runs in its own process and puts the reference checkout FIRST
    for name in ("ssn_models", "ops", "ops.ssn_ops", "model_zoo", "transforms"):
        if name in sys.modules and not getattr(sys.modules[name], "__file__", "").startswith(REF):
            raise ImportError("%s is already imported from %s: the reference arm needs its own process"
                              % (name, getattr(sys.modules[name], "__file__", "?")))
    sys.path.insert(0, REF)
    cwd = os.getcwd()
    os.chdir(REF)                      # pytorch_load.py:9 opens 'model_zoo/bninception/bn_inception.yaml' relative to the cwd
    try:
        import model_zoo.bninception.pytorch_load as pl
        pl.BNInception.load_state_dict = lambda self, sd, *a, **k: None
        import ssn_models
        import ops.ssn_ops as ssn_ops
    finally:
        os.chdir(cwd)
    _mods = (ssn_models, ssn_ops)
    return _mods


def build_model(num_class, modality, stpp_cfg, backbone_sd, heads_sd, test_mode=False):
    """reference SSN(BNInception, dropout=0, frozen BN) carrying the given synthetic weights"""
    import torch
    ssn_models, _ = import_reference()
    cwd = os.getcwd()
    os.chdir(REF)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            model = ssn_models.SSN(num_class, 2, 5, 2, modality, base_model="BNInception", dropout=0,
                                   stpp_cfg=stpp_cfg, test_mode=test_mode)
    finally:
        os.chdir(cwd)
    sd = model.state_dict()
    with torch.no_grad():
        for k, v in backbone_sd.items():
            sd["base_model." + k].copy_(v)
        for k, v in heads_sd.items():
            sd[k].copy_(v)
    return model


def train_step(model, batch, comp_w=0.1, reg_w=0.1):
    """one iteration of the reference's training loop body, ssn_train.py:207-236 (forward, three criteria, backward)"""
    import torch
    _, R = import_reference()
    x, sc, tgt, rtgt, ptype = batch
    act, act_t, comp, comp_t, reg, reg_l, reg_t = model(x, sc, tgt, rtgt, ptype)
    la = torch.nn.CrossEntropyLoss()(act, act_t)
    lc = R.CompletenessLoss()(comp, comp_t, 1, 7)          # fg_per_video = 1, fg + incomplete per video = 7 (ssn_train.py:189-190)
    lr = R.ClassWiseRegressionLoss()(reg, reg_l, reg_t)
    loss = la + comp_w * lc + reg_w * lr
    model.zero_grad()
    loss.backward()
    return float(loss), (float(la), float(lc), float(lr))
