"""CPU-side checks of the drop-in boundary: the C-ABI library builds/loads without a GPU and exports
every symbol include/vqa_b200.h declares; the host modules keep the reference's parameter layout."""
import os
import re
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared(debug=False):
    """Entry points declared by the header; the `#ifdef VQA_B200_DEBUG` section holds the debug-build-only hooks."""
    src = open(os.path.join(ROOT, "include", "vqa_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    dbg = re.findall(r"#ifdef VQA_B200_DEBUG(.*?)#endif", src, flags=re.S)
    if debug:
        src = "\n".join(dbg)
    else:
        src = re.sub(r"#ifdef VQA_B200_DEBUG.*?#endif", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(vqa_b200_\w+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from vqa_attention_networks_b200 import _lib
    lib = _lib.load()
    names = _declared()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), "missing export " + n
    assert set(names) == set(_lib.EXPORTED_SYMBOLS), set(names) ^ set(_lib.EXPORTED_SYMBOLS)
    assert lib.vqa_b200_abi_version() == 2


def test_release_library_has_no_global_state_hooks():
    """The hooks that write process-global state (descriptor overrides, cycle-counter buffers) exist in
    -DVQA_B200_DEBUG builds only; the shipped library must not export them (VERDICT r1, boundary)."""
    from vqa_attention_networks_b200 import _lib
    lib = _lib.load()
    dbg = _declared(debug=True)
    assert sorted(dbg) == sorted(_lib._DEBUG_PROTOTYPES)
    if os.environ.get("VQA_B200_DEBUG", "0") != "1":
        for n in dbg:
            assert not hasattr(lib, n), n + " exported by a release build"


def test_no_cpu_fallback():
    """The product path must fail loudly on CPU tensors instead of computing something else."""
    from vqa_attention_networks_b200 import Attention_layer, ops
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.pack_bf16(torch.zeros(4, 8))
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        Attention_layer(16, 1)(torch.zeros(2, 6, 16), torch.zeros(2, 5, 16))


def _cfg(**kw):
    base = dict(model_name="mhb_coAtt", q_vocab_size=20, emb_dim=6, hidden_dim=8, num_layers=1,
                img_feature_channel=16, img_feature_dim=6, a_vocab_size=7, glove=False)
    base.update(kw)
    return types.SimpleNamespace(**base)


@pytest.mark.parametrize("fixture,kind,kw", [
    ("mhbcoatt_eval", "mhbcoatt", {}),
    ("mhbcoatt_glove_eval", "mhbcoatt", {"glove": True}),
    ("mfb_eval", "mfb", {"model_name": "mfb"}),
    ("mfb_multilayer_eval", "mfb", {"model_name": "mfb-multilayer"}),
])
def test_state_dict_layout_matches_reference(fixture, kind, kw):
    """Parameter names, shapes and ranks are the reference's (recorded in the golden fixtures from the real
    modules): state dicts interchange and train_models.py:54-56's Xavier loop applies (every non-bias >= 2-D)."""
    from oracle import fixtures
    from vqa_attention_networks_b200 import MFB, MHBCoAtt
    rec = fixtures.load_fixture(fixture)
    shapes = {k: tuple(v) for k, v in rec["case"]["shapes"].items()}
    cfg = _cfg(**{**rec["case"]["cfg"], **kw}) if "cfg" in rec["case"] else _cfg(**kw)
    model = (MHBCoAtt if kind == "mhbcoatt" else MFB)(cfg)
    mine = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    assert mine == shapes
    for name, p in model.named_parameters():
        if name.find("bias") == -1:
            torch.nn.init.xavier_uniform_(p)          # must not raise
    model.load_state_dict(fixtures.make_params(rec["case"]["shapes"], 1), strict=True)


@pytest.mark.parametrize("fixture", ["hiecoatten_n4", "mhb_patched_eval", "attention_1_n2", "attention_2_n2",
                                     "attention_layer_1_n2", "attention_layer_2_n2", "nonlinear_layer_n2"])
def test_state_dict_layout_other_modules(fixture):
    """HieCoAtten / MHB / modules.py replacements: same parameter names and shapes as the real reference modules
    (shapes recorded by oracle/gen_golden.py), incl. the dead layers fc_Wbq and Attention_2.fc2."""
    from oracle import fixtures
    import vqa_attention_networks_b200 as V
    rec = fixtures.load_fixture(fixture)
    case = rec["case"]
    kind = case["model"]
    if kind == "hiecoatten":
        model = V.HieCoAtten(**case["ctor"])
    elif kind == "mhb":
        model = V.MHB(types.SimpleNamespace(**case["cfg"]))
    elif kind == "attention_1":
        model = V.Attention_1(case["D"])
    elif kind == "attention_2":
        model = V.Attention_2(case["D"])
    elif kind.startswith("attention_layer"):
        model = V.Attention_layer(case["D"], int(kind[-1]))
    else:
        model = V.Nonlinear_layer(case["D"])
    mine = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    assert mine == {k: tuple(v) for k, v in case["shapes"].items()}
    model.load_state_dict(fixtures.make_params(case["shapes"], 1), strict=True)


def test_networks_attentionnet_picks_up_the_modules():
    """networks.py:35-42 builds AttentionNet from modules.Attention_layer by name: the replacement must accept the
    same constructor call and register the same sub-module names (att_layer.fc.*)."""
    from vqa_attention_networks_b200 import Attention_layer
    layer = Attention_layer(512, 1)
    assert sorted(k for k, _ in layer.named_parameters()) == ["att_layer.fc.bias", "att_layer.fc.weight"]
    layer2 = Attention_layer(512, 2)
    assert sorted(k for k, _ in layer2.named_parameters()) == ["att_layer.fc1.weight", "att_layer.fc2.bias",
                                                               "att_layer.fc2.weight"]
    with pytest.raises(SystemExit):
        Attention_layer(512, 3)            # modules.py:19-20


def test_argument_validation_returns_error_codes_without_a_gpu():
    """The C ABI validates shapes / pointers before touching CUDA: negative status + a message, never a crash."""
    import ctypes
    from vqa_attention_networks_b200 import _lib
    L = _lib.load()
    null = ctypes.c_void_p(0)
    one = ctypes.c_void_p(16)          # non-null, never dereferenced on the host
    rc = L.vqa_b200_gemm(null, 0, 8, one, 0, 8, one, 0, 8, 4, 4, 8, None, None, 1, 0, 0, 0, None, 0, None, None)
    assert rc == -1 and b"gemm" in L.vqa_b200_last_error()
    rc = L.vqa_b200_gemm(one, 0, 8, one, 0, 8, one, 1, 8, 4, 4, 8, None, None, 1, 0, 1, 0, None, 0, None, None)
    assert rc == -1 and b"accumulate" in L.vqa_b200_last_error()          # accumulate needs an fp32 C
    rc = L.vqa_b200_mfb_fused(one, 8, one, 8, one, one, 8, 1, one, 0, 8, one, None, 1, 4, 30, 8, 0, None, None, 0.0, 0, None, None)
    assert rc == -1 and b"multiple of 20" in L.vqa_b200_last_error()      # k*o must keep the k=5 pools whole
    rc = L.vqa_b200_softmax_pool_fwd(one, 1, one, one, one, 2, 6, 16, 3, 0, None)
    assert rc == -1 and b"G must be 1 or 2" in L.vqa_b200_last_error()
    rc = L.vqa_b200_softmax_pool_fwd(one, 1, one, one, one, 2, 6, 12, 2, 0, None)
    assert rc == -2                                                        # D not a multiple of the 16-byte vector
    rc = L.vqa_b200_mfb_bwd(one, 1, 8, one, 0, 8, one, one, one, 8, one, 1, one, 1, one, one, 1, 4, 5000, 0, None, None, None, 0.0, 0, None, None)
    assert rc == -1 and b"share a dtype" in L.vqa_b200_last_error()
    rc = L.vqa_b200_lstm_cell_fwd(one, None, one, one, 1024, one, 64, 1022, 1, 0, 0.0, 0, None, None)
    assert rc == -1 and b"lstm_cell_fwd" in L.vqa_b200_last_error()       # H must be a multiple of 4
    rc = L.vqa_b200_lstm_cell_fwd(one, None, one, one, 1024, ctypes.c_void_p(20), 64, 1024, 1, 0, 0.0, 0, None, None)
    assert rc == -2                                                        # bf16 h_t rows: 8-byte aligned
    rc = L.vqa_b200_lstm_cell_bwd(one, None, one, one, 512, one, one, one, 64, 1024, 0, 0.0, 0, None, None)
    assert rc == -1 and b"lstm_cell_bwd" in L.vqa_b200_last_error()       # row pitch of dout shorter than H
    rc = L.vqa_b200_lstm_fwd(one, one, one, one, None, 4, 26, 1024, 1.5, 0, None, None)
    assert rc == -1 and b"dropout" in L.vqa_b200_last_error()
    with pytest.raises(RuntimeError, match="status -1"):
        _lib.check(-1, "gemm")


def test_every_kernel_entry_point_is_a_torch_custom_op():
    """SURVEY 8b / north_star: "a thin C-ABI torch custom-op extension".  Each kernel entry point of the header is one
    dispatcher op torch.ops.vqa_b200.<name> whose schema mirrors the C prototype (pointers -> Tensor?, the written ones
    declared as mutated, the stream implicit); only the pure queries and the pointer-table Adam entry points stay plain
    C calls."""
    from vqa_attention_networks_b200 import _lib, ops
    ops._register_custom_ops()
    declared = set(_declared())
    wrapped = set(_lib.MUTATED_ARGS)
    assert wrapped <= declared
    assert declared - wrapped == {"vqa_b200_abi_version", "vqa_b200_last_error", "vqa_b200_lstm_supported",
                                  "vqa_b200_adam_step", "vqa_b200_adam_step_dev"}
    for name, mutated in _lib.MUTATED_ARGS.items():
        op = getattr(torch.ops.vqa_b200, name[len("vqa_b200_"):]).default
        schema = op._schema
        argtypes = _lib._PROTOTYPES[name][1]
        assert len(schema.arguments) == len(argtypes) - 1                     # the stream is not an argument
        assert len(schema.returns) == 0
        for i, a in enumerate(schema.arguments):
            is_ptr = argtypes[i].__name__ == "c_void_p"
            assert (str(a.type) == "Optional[Tensor]") == is_ptr, (name, i, str(a.type))
            assert bool(a.alias_info is not None and a.alias_info.is_write) == (i in mutated), (name, i)
    # CPU tensors have no kernel: the dispatcher refuses instead of computing something else
    with pytest.raises((NotImplementedError, RuntimeError)):
        torch.ops.vqa_b200.inv_norm(torch.ones(4), torch.zeros(4), 4)


def test_ctypes_prototypes_match_the_header():
    """Every prototype in _lib._PROTOTYPES (the source of the ctypes bindings AND of the custom-op schemas) must agree
    with the declaration in include/vqa_b200.h: same number of parameters, pointers where the header has pointers,
    64-bit integers where it has int64_t, floats / doubles / 32-bit integers likewise.  A drifted prototype would still
    load and silently pass garbage."""
    import ctypes
    from vqa_attention_networks_b200 import _lib
    src = open(os.path.join(ROOT, "include", "vqa_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"//[^\n]*", "", src)
    decls = dict((m.group(1), m.group(2)) for m in re.finditer(r"\b(vqa_b200_\w+)\s*\(([^;{]*?)\)\s*;", src, flags=re.S))
    kinds = {ctypes.c_void_p: "ptr", ctypes.c_char_p: "ptr", ctypes.c_int: "i32", ctypes.c_uint32: "u32",
             ctypes.c_int64: "i64", ctypes.c_float: "f32", ctypes.c_double: "f64"}

    def kind_of(param):
        p = " ".join(param.split())
        if "*" in p:
            return "ptr"
        for pat, k in ((r"\bint64_t\b", "i64"), (r"\buint32_t\b", "u32"), (r"\bdouble\b", "f64"), (r"\bfloat\b", "f32"),
                       (r"\bint\b", "i32")):
            if re.search(pat, p):
                return k
        raise AssertionError("unrecognised parameter type: " + p)

    checked = 0
    for name, (restype, argtypes) in _lib._PROTOTYPES.items():
        if name not in decls:
            continue                                   # debug-only hooks
        params = [p for p in decls[name].split(",") if p.strip() and p.strip() != "void"]
        assert len(params) == len(argtypes), (name, len(params), len(argtypes))
        for i, (p, a) in enumerate(zip(params, argtypes)):
            assert kind_of(p) == kinds[a], (name, i, p.strip(), a.__name__)
        checked += 1
    assert checked >= 30
