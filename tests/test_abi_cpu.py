"""CPU-only checks of the drop-in boundary: the C-ABI library builds/loads without a GPU, exports every symbol that
include/klab_b200.h declares (with the declared arity), refuses to compute without an sm_100 device (no CPU fallback), and
the Python module trees carry the reference's (HuggingFace) state-dict key layout."""
import ctypes as C
import os
import re
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_prototypes():
    h = open(os.path.join(ROOT, "include", "klab_b200.h")).read()
    h = re.sub(r"/\*.*?\*/", "", h, flags=re.S)
    return re.findall(r"(?:int|long long|const char\*)\s+(klab_\w+)\s*\(([^;]*?)\)\s*;", h, flags=re.S)


def test_library_exports_every_declared_symbol():
    from klab_multimodalmodel_b200 import _lib as L
    lib = L.lib()
    protos = header_prototypes()
    assert len(protos) >= 30
    for name, args in protos:
        assert hasattr(lib, name), f"{name} declared in klab_b200.h but not exported"
        n = 0 if args.strip() in ("void", "") else len(args.split(","))
        assert name in L.SIGNATURES, f"{name} has no ctypes signature"
        assert len(L.SIGNATURES[name]) == n, f"{name}: header has {n} arguments, binding has {len(L.SIGNATURES[name])}"
    assert set(L.SIGNATURES) == {n for n, _ in protos}
    assert lib.klab_abi_version() == 1


def test_ctypes_argument_types_match_header():
    from klab_multimodalmodel_b200 import _lib as L
    scalar = {"int": C.c_int, "long long": C.c_longlong, "float": C.c_float, "unsigned long long": C.c_ulonglong, "double": C.c_double}
    for name, args in header_prototypes():
        if args.strip() in ("void", ""):
            continue
        for i, (a, bound) in enumerate(zip(args.split(","), L.SIGNATURES[name])):
            a = a.strip()
            if "*" in a:
                want = C.POINTER(L.GemmEpilogue) if "klab_gemm_epilogue" in a else C.c_void_p
            else:
                want = scalar[a.rsplit(" ", 1)[0].strip()]
            assert want is bound, f"{name} arg {i} ({a})"


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a box without a GPU")
def test_no_cpu_fallback():
    from klab_multimodalmodel_b200 import _lib as L
    from klab_multimodalmodel_b200 import ops as O
    lib = L.lib()
    assert lib.klab_check_device() == 3                      # KLAB_ERR_UNSUPPORTED
    assert b"no CPU fallback" in lib.klab_last_error()
    e = L.GemmEpilogue()
    assert lib.klab_gemm(None, L.F32, 4, 4, 4, None, 4, 0, None, 4, 0, None, 4, C.byref(e)) == 3
    from klab_multimodalmodel_b200.modeling import Swinv2Config, T5Config
    from klab_multimodalmodel_b200.models.model import MyModel
    tcfg = T5Config(vocab_size=64, d_model=128, d_ff=64, num_layers=1, num_heads=2)
    scfg = Swinv2Config(image_size=32, embed_dim=32, depths=(1, 1, 1), num_heads=(1, 2, 4), window_size=4, pretrained_window_sizes=(0, 0, 0))
    args = types.SimpleNamespace(result_dir="/tmp", language_model_name=tcfg, image_model_name=scfg, image_model_train=False,
                                 transformer_model_name=tcfg)
    model = MyModel(args)
    with pytest.raises(RuntimeError, match="no CPU path"):
        model({"pixel_values": torch.randn(1, 3, 32, 32)}, {"input_ids": torch.ones(1, 4, dtype=torch.long)},
              {"input_ids": torch.ones(1, 4, dtype=torch.long)})


def test_state_dict_layout_matches_reference_keys():
    from klab_multimodalmodel_b200.modeling import Swinv2Config, Swinv2Model, T5Config, T5EncoderModel, T5ForConditionalGeneration
    from oracle.caption_model import swin_param_shapes, t5_param_shapes
    from oracle.swinv2 import SwinDims
    from oracle.t5 import T5Dims
    kw = dict(vocab_size=512, d_model=128, d_ff=256, num_layers=2, num_heads=2)
    for cls, enc_only in ((T5ForConditionalGeneration, False), (T5EncoderModel, True)):
        sd = cls(T5Config(**kw)).state_dict()
        ref = t5_param_shapes(T5Dims(**kw), encoder_only=enc_only)
        assert set(sd) == set(ref)
        assert all(tuple(sd[k].shape) == tuple(ref[k]) for k in ref)
    skw = dict(image_size=64, embed_dim=32, depths=(2, 2, 2), num_heads=(1, 2, 4), window_size=4, pretrained_window_sizes=(0, 0, 0))
    sd = Swinv2Model(Swinv2Config(**skw)).state_dict()
    ref = swin_param_shapes(SwinDims(**skw))
    assert set(sd) == set(ref) and all(tuple(sd[k].shape) == tuple(ref[k]) for k in ref)
    t = T5ForConditionalGeneration(T5Config(**kw))
    assert t.lm_head.weight is t.shared.weight and t.decoder.embed_tokens.weight is t.shared.weight   # tied (modeling_t5.py:956-960)


def test_state_dict_layout_matches_transformers_if_present():
    """Against the layout transformers 5.5.0 stored in tests/golden/hf_layout.json (tests/golden/make_hf_golden.py), and
    against the installed transformers classes where they import."""
    import json

    from klab_multimodalmodel_b200.modeling import Swinv2Config, Swinv2Model, T5Config, T5ForConditionalGeneration
    from tests.golden.make_hf_golden import LAYOUT_SWIN, LAYOUT_T5
    ours = T5ForConditionalGeneration(T5Config(**LAYOUT_T5))
    sw = Swinv2Model(Swinv2Config(**LAYOUT_SWIN, pretrained_window_sizes=(0, 0, 0)))
    with open(os.path.join(ROOT, "tests", "golden", "hf_layout.json")) as fh:
        stored = json.load(fh)
    for model, layout in ((ours, stored["t5"]), (sw, stored["swin"])):
        assert set(layout) == set(model.state_dict())
        model.load_state_dict({k: torch.zeros(shape) for k, shape in layout.items()}, strict=True)
    try:
        import transformers
    except ImportError:
        return
    hf = transformers.T5ForConditionalGeneration(transformers.T5Config(vocab_size=512, d_model=128, d_kv=64, d_ff=256, num_layers=2,
                                                                       num_heads=2, decoder_start_token_id=0))
    assert set(hf.state_dict()) == set(ours.state_dict())
    ours.load_state_dict(hf.state_dict(), strict=True)
    hfs = transformers.Swinv2Model(transformers.Swinv2Config(image_size=64, embed_dim=32, depths=[2, 2, 2], num_heads=[1, 2, 4], window_size=4))
    assert set(hfs.state_dict()) == set(sw.state_dict())
    sw.load_state_dict(hfs.state_dict(), strict=True)


def test_t5_bucket_lut_and_swin_tables_match_oracle():
    from klab_multimodalmodel_b200 import ops as O
    from oracle import swinv2 as osw
    from oracle import t5 as ot5
    for bidir in (True, False):
        lut, rz = O.t5_rel_bucket_lut(200, 300, bidir, 32, 128)
        assert rz == 199 and torch.equal(lut.long(), ot5.relative_position_bucket(torch.arange(-199, 300), bidir, 32, 128))
    for w, pw in ((7, 0), (8, 0), (12, 8)):
        coords, index = O.swin_tables(w, pw)
        assert torch.equal(index.long(), osw.position_index(w)) and torch.allclose(coords, osw.coords_table(w, pw))
