"""CPU: libmmg.so builds for sm_100a, loads without a GPU/driver, exports every symbol include/mmg.h declares, and the
ctypes mirror of every argument block has the C struct's size.  No compute calls here."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_header_symbols():
    from muse_maskgit_pytorch_b200 import build, _lib
    build.build()
    header = open(os.path.join(ROOT, "include", "mmg.h")).read()
    declared = set(re.findall(r"^\s*(?:int|int64_t|uint64_t|const char\*)\s+(mmg_[a-z0-9_]+)\s*\(", header, re.M))
    assert {"mmg_linear", "mmg_attention", "mmg_logits_sample", "mmg_vq_lfq_encode", "mmg_vq_l2_argmin", "mmg_conv2d",
            "mmg_conv_transpose2d", "mmg_remask", "mmg_version"} <= declared
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in mmg.h but not exported"
    assert set(_lib.EXPORTS) | set(_lib.PLAIN_EXPORTS) == declared
    assert _lib.lib().mmg_version() == 100          # also runs the struct-size self check


def test_ops_fail_loudly_without_library(monkeypatch, tmp_path):
    from muse_maskgit_pytorch_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "missing.so"))
    try:
        _lib.lib()
    except _lib.MMGError as e:
        assert "no fallback" in str(e)
    else:
        raise AssertionError("missing library must raise")


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "muse_maskgit_pytorch_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in src.replace("# oracle", ""), f"{fn} references the oracle"


def test_state_dict_keys_match_reference_tables():
    """Checkpoint-key contract (SURVEY.md 8b): our parameter holders expose exactly the reference's keys/shapes
    (oracle/shapes.py is asserted against the unmodified reference in tests/golden/make_golden.py)."""
    import muse_maskgit_pytorch_b200 as M
    from muse_maskgit_pytorch_b200 import t5
    from oracle import shapes
    t5.T5_CONFIGS["synth-96"] = {"d_model": 96}
    tr = M.MaskGitTransformer(num_tokens=1024, dim=128, seq_len=16, depth=2, heads=2, t5_name="synth-96")
    got = {k: tuple(v.shape) for k, v in tr.state_dict().items()}
    assert got == {k: tuple(v) for k, v in shapes.transformer_shapes(1024, 128, 16, 2, heads=2, text_dim=96).items()}
    vae = M.VQGanVAE(dim=64, codebook_size=512)
    got = {k: tuple(v.shape) for k, v in vae.state_dict().items() if k != "quantizer.mask"}
    assert got == {k: tuple(v) for k, v in shapes.vae_shapes(64, codebook_size=512).items()}
    assert "quantizer.mask" in vae.state_dict()
    critic = M.TokenCritic(num_tokens=1024, dim=128, seq_len=16, depth=1, heads=2, t5_name="synth-96")
    assert critic.state_dict()["to_logits.weight"].shape == (1, 128) and critic.mask_id is None


def test_decode_step_workspace_query_is_host_only():
    """mmg_decode_step_workspace_bytes is pure host arithmetic: callable without a GPU, grows with the logits buffer."""
    from muse_maskgit_pytorch_b200 import _lib
    f = _lib.lib().mmg_decode_step_workspace_bytes
    c3 = f(64, 2, 256, 512, 8, 1408, 65536, 256)
    assert c3 >= 64 * 256 * 65536 * 4 and c3 % 256 == 0
    assert f(8, 2, 256, 512, 8, 1408, 65536, 256) < c3 and f(0, 2, 256, 512, 8, 1408, 65536, 256) == 0


def test_baseline_ref_is_the_unmodified_reference():
    """baseline/_ref (the reference arm of bench.py) holds the unmodified reference: its modules are exactly those of the upstream package,
    byte for byte, by the SHA-256 digests recorded from the upstream sources in tests/golden/reference_sources.json (make_golden.py)."""
    import hashlib
    import json
    import pytest
    inst = os.path.join(ROOT, "baseline", "_ref", "muse_maskgit_pytorch")
    if not os.path.isdir(inst):
        pytest.skip("baseline/_ref is not installed (build() installs it only where the reference sources are available)")
    want = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_sources.json")))
    got = {f: hashlib.sha256(open(os.path.join(inst, f), "rb").read()).hexdigest() for f in os.listdir(inst) if f.endswith(".py")}
    assert want and got == want, sorted(f for f in set(got) | set(want) if got.get(f) != want.get(f))


def test_pack_cache_digest_tracks_weights():
    """The on-disk pre-pack cache key (pack_cache.weights_digest) is a function of names, shapes, dtypes and bytes of the module's tensors."""
    import torch
    from muse_maskgit_pytorch_b200 import pack_cache
    torch.manual_seed(0)
    a, b = torch.nn.Linear(8, 4), torch.nn.Linear(8, 4)
    b.load_state_dict(a.state_dict())
    assert pack_cache.weights_digest(a, ("bf16",)) == pack_cache.weights_digest(b, ("bf16",))
    assert pack_cache.weights_digest(a, ("bf16",)) != pack_cache.weights_digest(a, ("fp32",))
    with torch.no_grad():
        b.weight[0, 0] += 1e-3
    assert pack_cache.weights_digest(a, ("bf16",)) != pack_cache.weights_digest(b, ("bf16",))
