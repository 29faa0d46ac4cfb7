"""CPU-side tests: the C-ABI library loads and exports every symbol include/ssnb.h declares, the
host-side tables agree with the oracle, and argument validation works without a GPU."""
import ctypes as C
import os
import re

import pytest
import torch

from oracle import ssn_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from ssn_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "ssnb.h")).read()
    declared = set(re.findall(r"\b(ssnb_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(_lib.lib, name), "libssn_b200.so does not export " + name
    assert declared == set(_lib.SIGNATURES), (declared ^ set(_lib.SIGNATURES))


def test_conv_table_matches_oracle():
    from ssn_b200.engine import conv_table
    for cin in (3, 10):
        assert conv_table(cin) == [tuple(r) for r in O.conv_layers(cin)]


def test_engine_plan_without_gpu():
    from ssn_b200 import _lib
    cfg = _lib.Config(3, 18, _lib.EXACT_FP32, 1, 1.0)
    h = C.c_void_p()
    _lib.check(_lib.lib.ssnb_create(C.byref(cfg), C.byref(h)))
    assert _lib.lib.ssnb_workspace_bytes(h) > 0
    n = _lib.lib.ssnb_num_ops(h)
    assert n == 69 + 13        # 69 convs, 12 spatial pools + global pool
    shape = [C.c_int() for _ in range(3)]
    _lib.check(_lib.lib.ssnb_value_shape(h, b"inception_4e_output", *[C.byref(s) for s in shape]), h)
    assert [s.value for s in shape] == [1056, 7, 7]
    assert _lib.lib.ssnb_value_shape(h, b"nonexistent", None, None, None) != 0
    assert b"unknown value" in _lib.lib.ssnb_last_error(h)
    # calls that need device state fail with an error code, not a crash
    assert _lib.lib.ssnb_backbone_fwd(h, None, None, None) != 0
    _lib.lib.ssnb_destroy(h)
    bad = _lib.Config(3, 0, 0, 0, 1.0)
    assert _lib.lib.ssnb_create(C.byref(bad), C.byref(h)) != 0


def test_module_surface_matches_reference(golden_dir):
    import json
    import ssn_models
    m = ssn_models.SSN(20, 2, 5, 2, "RGB", base_model="BNInception", dropout=0.8)
    assert sum(p.numel() for p in m.parameters()) == 10599025          # SURVEY §8c
    g = json.load(open(os.path.join(golden_dir, "bninception_graph.json")))
    ref_keys = ["base_model." + k for k in g["state_dict_keys"] if not k.startswith("fc.")]
    mine = [k for k in m.state_dict().keys() if k.startswith("base_model.")]
    assert mine == ref_keys
    assert isinstance(m.base_model.fc, torch.nn.Dropout)
    pol = m.get_optim_policies()
    assert [len(p["params"]) for p in pol] == [1, 1, 71, 71, 0]
    assert [(p["lr_mult"], p["decay_mult"]) for p in pol] == [(1, 1), (2, 0), (1, 1), (2, 0), (1, 0)]
    m.train()
    assert all(not b.training for b in m.base_model.modules() if isinstance(b, torch.nn.BatchNorm2d))
    assert (m.crop_size, m.scale_size, m.input_mean, m.input_std) == (224, 256, [104, 117, 128], [1])
    with pytest.raises(ValueError):
        ssn_models.SSN(20, 2, 5, 2, "RGB", base_model="nope")
    with pytest.raises(RuntimeError):          # no CPU fallback: fails loudly
        m(torch.zeros(2, 8 * 9 * 3, 224, 224), torch.zeros(2, 8, 2), torch.zeros(2, 8).long(), torch.zeros(2, 8, 2),
          torch.zeros(2, 8).long())


def test_stpp_part_table_matches_oracle():
    from ops.ssn_ops import StructuredTemporalPyramidPooling
    for cfg, seg in (((1, (1, 2), 1), [2, 7, 9]), ([1, 1, 1], [2, 7, 9]), (((1, 2), (1, 2, 4), 2), [4, 12, 16]),
                     ((1, (1, 2), 1), [1, 2, 3])):
        mod = StructuredTemporalPyramidPooling(1024, True, configs=cfg)
        lo, hi, nm, col = mod.part_table(seg)
        assert list(zip(lo, hi, nm, col)) == O.stpp_parts(cfg, seg)
    with pytest.raises(ValueError):
        StructuredTemporalPyramidPooling(8, True, configs=("x", 1, 1))


def test_bench_reference_arm_prints_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours) prints ONE JSON line with the contract keys."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0",
                          "--videos-per-gpu", "2"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "proposals/s" and d["higher_is_better"] is True and d["value"] > 0
    # kind: the unmodified reference when SSNB_REFERENCE_DIR names a checkout of it, else the oracle port
    ref = os.environ.get("SSNB_REFERENCE_DIR")
    has_ref = bool(ref) and os.path.exists(os.path.join(ref, "ssn_models.py"))
    assert d["cpu_baseline"]["kind"] == ("reference" if has_ref else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"] and d["steps"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "proposals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_clock_sampler_survives_a_box_without_gpu():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    with bench.ClockSampler(0) as cs:
        pass
    s = cs.summary()
    assert set(s) >= {"sm_mhz", "sm_max_mhz", "reasons", "samples"} and isinstance(s["reasons"], list)
    assert bench.usable_cores() >= 1


def test_flow_model_conv1_is_mean_expanded():
    """a4: SSN(modality='Flow') builds the 3-channel net and swaps conv1 for the 10-channel kernel that repeats the mean of
    the RGB kernels over the input channels, bias kept (_construct_flow_model, ssn_models.py:318-343).  No GPU needed."""
    import ssn_models
    import model_zoo
    torch.manual_seed(5)
    rgb = model_zoo.BNInception(in_channels=3)
    w3, b3 = rgb.conv1_7x7_s2.weight.data.clone(), rgb.conv1_7x7_s2.bias.data.clone()
    torch.manual_seed(5)
    m = ssn_models.SSN(4, 2, 5, 2, "Flow", base_model="BNInception", dropout=0)
    c1 = m.base_model.conv1_7x7_s2
    assert tuple(c1.weight.shape) == (64, 10, 7, 7) and c1.in_channels == 10 and m.base_model.in_channels() == 10
    assert torch.equal(c1.bias.data, b3)
    mean = w3.mean(dim=1, keepdim=True)
    for ch in range(10):
        assert torch.equal(c1.weight.data[:, ch:ch + 1], mean)
    assert m.input_mean == [128] and m.new_length == 5
    assert "base_model.conv1_7x7_s2.weight" in m.state_dict() and m.state_dict()["base_model.conv1_7x7_s2.weight"].shape[1] == 10


def test_header_is_plain_c_and_ctypes_mirrors_its_structs(tmp_path):
    """include/ssnb.h must compile as C99 on its own (it is the drop-in boundary: no C++ or torch types), and the ctypes
    mirrors in ssn_b200/_lib.py must have the same size and field offsets as the C structs."""
    import shutil
    import subprocess
    from ssn_b200 import _lib
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    hdr = open(os.path.join(ROOT, "include", "ssnb.h")).read()

    def fields(struct):            # field names of `typedef struct { ... } <struct>;` in declaration order
        body = re.search(r"typedef struct \{([^{}]*)\}\s*" + struct + ";", hdr).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        names = []
        for decl in body.split(";"):
            decl = decl.strip()
            if decl:
                names += [re.sub(r"\[.*\]", "", n).strip() for n in decl.split(None, 1)[1].split(",")]
        return names

    structs = {"ssnb_config": _lib.Config, "ssnb_heads_cfg": _lib.HeadsCfg}
    prints = []
    for s in structs:
        prints.append('printf("%s %%zu\\n", sizeof(%s));' % (s, s))
        prints += ['printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (s, f, s, f) for f in fields(s)]
    src = tmp_path / "abi.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ssnb.h"\nint main(void) { %s return 0; }\n' % " ".join(prints))
    exe = tmp_path / "abi"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    c_layout = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for s, mirror in structs.items():
        assert int(c_layout[s]) == C.sizeof(mirror), s
        c_offsets = {f: int(c_layout["%s.%s" % (s, f)]) for f in fields(s)}
        assert [name for name, _ in mirror._fields_] == list(c_offsets), (s, list(c_offsets))
        for name, _ in mirror._fields_:
            assert getattr(mirror, name).offset == c_offsets[name], (s, name)
