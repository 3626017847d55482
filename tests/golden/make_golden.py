"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference):   python tests/golden/make_golden.py
The reference's four missing third-party packages are replaced by the stand-ins in tests/golden/_shims
(see SURVEY.md section 8c / Appendix A); everything else is the reference's own code.  Weights and inputs
come from oracle/synth.py (hash-keyed on the parameter name) so tests can regenerate them anywhere.
The .npz files written here are committed; this script documents how they were made.
"""
import os
import sys
import json
import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

import transformers  # noqa: F401  (must be imported BEFORE the accelerate stand-in is visible)
from transformers import T5Config

sys.path.insert(0, os.path.join(HERE, "_shims"))
sys.path.insert(0, "/root/reference")

from muse_maskgit_pytorch import t5 as ref_t5                      # noqa: E402
from muse_maskgit_pytorch import VQGanVAE, MaskGitTransformer, MaskGit   # noqa: E402
from muse_maskgit_pytorch.muse_maskgit_pytorch import cosine_schedule    # noqa: E402
import math                                                         # noqa: E402

from oracle import synth, shapes                                    # noqa: E402

torch.set_grad_enabled(False)


def seed_t5(name, d_model):
    ref_t5.T5_CONFIGS[name] = dict(config=T5Config(d_model=d_model))


def fill(module, table, seed):
    sd = module.state_dict()
    got = {k: tuple(v.shape) for k, v in sd.items() if not k.startswith("discr.") and k != "quantizer.mask"}
    want = {k: tuple(v) for k, v in table.items()}
    assert got == want, (sorted(set(got) ^ set(want)), [(k, got[k], want[k]) for k in got if k in want and got[k] != want[k]])
    vals = synth.fill_state_dict(table, seed=seed)
    for k, v in vals.items():
        sd[k].copy_(torch.from_numpy(v))
    return {k: torch.from_numpy(v) for k, v in vals.items()}


def text_embeds(name, b, m, d, seed):
    te = torch.from_numpy(synth.normal(name, (b, m, d), seed))
    te[1::2, (3 * m) // 4:] = 0.          # padding rows on odd batch entries (exercises context_mask)
    return te


def save(name, **arrs):
    out = {k: (v.numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in arrs.items()}
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, {k: v.shape for k, v in out.items()})


# ------------------------------------------------------------------ schedules / top-k counts (known answers)
def schedule(seq, T):
    return [max(int((cosine_schedule(t) * seq).item()), 1) for t in torch.linspace(0, 1, T)]


known = dict(
    sched_256_18=schedule(256, 18), sched_1024_18=schedule(1024, 18), sched_16_18=schedule(16, 18),
    sched_16_6=schedule(16, 6), sched_64_8=schedule(64, 8),
    topk={str(v): math.ceil((1 - 0.9) * v) for v in (512, 1024, 8192, 65536)},
)
assert known["sched_256_18"] == [256, 254, 251, 246, 238, 229, 217, 204, 189, 172, 154, 134, 114, 92, 70, 47, 23, 1]
with open(os.path.join(HERE, "known_answers.json"), "w") as f:
    json.dump(known, f, indent=1)

# ------------------------------------------------------------------ SHA-256 of the reference's modules (tests/test_abi.py checks baseline/_ref against them)
import hashlib                                                      # noqa: E402
pkg_dir = os.path.dirname(os.path.abspath(ref_t5.__file__))
with open(os.path.join(HERE, "reference_sources.json"), "w") as f:
    json.dump({n: hashlib.sha256(open(os.path.join(pkg_dir, n), "rb").read()).hexdigest() for n in sorted(os.listdir(pkg_dir)) if n.endswith(".py")},
              f, indent=1)

# ------------------------------------------------------------------ G1: config C1 — VAE dim=64 cb=512 on 4x3x32x32
vae = VQGanVAE(dim=64, codebook_size=512).eval()
fill(vae, shapes.vae_shapes(64, codebook_size=512), seed=11)
img = torch.from_numpy(synth.uniform("c1.img", (4, 3, 32, 32), 11))
fq, ids, _ = vae.encode(img)
rec = vae.decode_from_ids(ids)
rec2 = vae(img)
assert torch.equal(rec, rec2) or (rec - rec2).abs().max() < 1e-6
fmap = vae.enc_dec.encode(img)
proj = vae.quantizer.project_in(fmap.permute(0, 2, 3, 1))
save("vae_c1", ids=ids.long(), recon=rec, fmap=fmap, proj=proj, fmap_q=fq)

# ------------------------------------------------------------------ G2: small VAE (dim=16, layers=2, cb=1024) 2x3x16x16
vae_s = VQGanVAE(dim=16, layers=2, codebook_size=1024).eval()
fill(vae_s, shapes.vae_shapes(16, layers=2, codebook_size=1024), seed=12)
img = torch.from_numpy(synth.uniform("g2.img", (2, 3, 16, 16), 12))
fq, ids, _ = vae_s.encode(img)
save("vae_small", ids=ids.long(), recon=vae_s.decode_from_ids(ids), fmap=vae_s.enc_dec.encode(img), fmap_q=fq)

# ------------------------------------------------------------------ G3: small transformer forward (cond / null / CFG)
for tag, d_text, flash in (("tr_small", 128, False), ("tr_small_proj", 96, False), ("tr_small_flash", 128, True)):
    seed_t5(f"synth-{d_text}", d_text)
    tr = MaskGitTransformer(num_tokens=1024, dim=128, seq_len=16, depth=2, dim_head=64, heads=2,
                            t5_name=f"synth-{d_text}", flash=flash).eval()
    fill(tr, shapes.transformer_shapes(1024, 128, 16, 2, heads=2, text_dim=d_text), seed=13)
    ids = torch.from_numpy((synth.uniform("g3.ids", (3, 16), 13) * 1025).astype(np.int64))
    ids[:, ::3] = 1024
    te = text_embeds("g3.te", 3, 8, d_text, 13)
    lc, emb = tr(ids, text_embeds=te, return_embed=True)
    ln_ = tr(ids, text_embeds=te, cond_drop_prob=1.)
    cfg = tr.forward_with_cond_scale(ids, text_embeds=te, cond_scale=3.)
    if tag == "tr_small":
        save(tag, ids=ids, logits_cond=lc, logits_null=ln_, logits_cfg=cfg, embed=emb)
    else:
        save(tag, ids=ids, logits_cfg=cfg, embed=emb)

# ------------------------------------------------------------------ G4: base generate, small (fmap 4x4, V=1024)
seed_t5("synth-128", 128)
tr = MaskGitTransformer(num_tokens=1024, dim=128, seq_len=16, depth=2, dim_head=64, heads=2,
                        t5_name="synth-128", flash=False).eval()
fill(tr, shapes.transformer_shapes(1024, 128, 16, 2, heads=2, text_dim=128), seed=13)
vae_s = VQGanVAE(dim=16, layers=2, codebook_size=1024).eval()
fill(vae_s, shapes.vae_shapes(16, layers=2, codebook_size=1024), seed=12)
mg = MaskGit(image_size=16, transformer=tr, vae=vae_s).eval()
te = text_embeds("g4.te", 3, 8, 128, 14)
tr.encode_text = lambda texts: te
for T in (6, 18):
    torch.manual_seed(777)
    u_probe = torch.zeros(7).uniform_(0, 1)
    torch.manual_seed(777)
    grabbed = {}
    orig = mg.vae.decode_from_ids
    mg.vae.decode_from_ids = lambda ids_, _o=orig, _g=grabbed: (_g.__setitem__("ids", ids_.clone()), _o(ids_))[1]
    images = mg.generate(texts=["a"] * 3, timesteps=T, cond_scale=3., temperature=1.)
    mg.vae.decode_from_ids = orig
    save(f"gen_small_T{T}", images=images, ids=grabbed["ids"], u_probe=u_probe)

# ------------------------------------------------------------------ G5: super-res generate, small (cond 16x16 -> 32x32; fmap 8x8, 16 cond tokens)
tr2 = MaskGitTransformer(num_tokens=1024, dim=128, seq_len=64, depth=2, dim_head=64, heads=2,
                         t5_name="synth-128", flash=False).eval()
fill(tr2, shapes.transformer_shapes(1024, 128, 64, 2, heads=2, text_dim=128), seed=15)
mg2 = MaskGit(image_size=32, transformer=tr2, vae=vae_s, cond_image_size=16).eval()
tr2.encode_text = lambda texts: te[:2]
cond = torch.from_numpy(synth.uniform("g5.cond", (2, 3, 16, 16), 15))
torch.manual_seed(778)
grabbed = {}
orig = mg2.vae.decode_from_ids
mg2.vae.decode_from_ids = lambda ids_, _o=orig, _g=grabbed: (_g.__setitem__("ids", ids_.clone()), _o(ids_))[1]
images = mg2.generate(texts=["a"] * 2, cond_images=cond, timesteps=8)
mg2.vae.decode_from_ids = orig
_, cond_ids, _ = mg2.cond_vae.encode(cond)
save("gen_superres_small", images=images, ids=grabbed["ids"], cond_ids=cond_ids.long())

# ------------------------------------------------------------------ G6-G8: generate()'s optional branches (SURVEY.md 8f #3)
from muse_maskgit_pytorch import TokenCritic                        # noqa: E402


def run_generate(mg_, T, seed, **kw):
    torch.manual_seed(seed)
    g = {}
    orig_ = mg_.vae.decode_from_ids
    mg_.vae.decode_from_ids = lambda ids_, _o=orig_, _g=g: (_g.__setitem__("ids", ids_.clone()), _o(ids_))[1]
    images_ = mg_.generate(texts=["a"] * 3, timesteps=T, cond_scale=3., temperature=1., **kw)
    mg_.vae.decode_from_ids = orig_
    return images_, g["ids"]


# G6: self-conditioning (muse_maskgit_pytorch.py:325-328, 574)
tr_sc = MaskGitTransformer(num_tokens=1024, dim=128, seq_len=16, depth=2, dim_head=64, heads=2,
                           t5_name="synth-128", flash=False, self_cond=True).eval()
fill(tr_sc, shapes.transformer_shapes(1024, 128, 16, 2, heads=2, text_dim=128), seed=21)
tr_sc.encode_text = lambda texts: te
mg_sc = MaskGit(image_size=16, transformer=tr_sc, vae=vae_s).eval()
images, ids = run_generate(mg_sc, 8, 779)
save("gen_selfcond_small", images=images, ids=ids)

# G7: separate token critic (muse_maskgit_pytorch.py:383-386, 590-600)
critic = TokenCritic(num_tokens=1024, dim=128, seq_len=16, depth=1, dim_head=64, heads=2, t5_name="synth-128", flash=False).eval()
fill(critic, shapes.transformer_shapes(1024, 128, 16, 1, heads=2, text_dim=128, add_mask_id=False, dim_out=1), seed=22)
critic.encode_text = lambda texts: te
mg_tc = MaskGit(image_size=16, transformer=tr, vae=vae_s, token_critic=critic).eval()
tr.encode_text = lambda texts: te
images, ids = run_generate(mg_tc, 8, 780, critic_noise_scale=0.7)
save("gen_critic_small", images=images, ids=ids)
images, ids = run_generate(mg_tc, 8, 780, force_not_use_token_critic=True)
save("gen_critic_forced_off_small", images=images, ids=ids)

# G8: self token critic on a self-conditioned transformer (muse_maskgit_pytorch.py:352-361, 475-476)
mg_self = MaskGit(image_size=16, transformer=tr_sc, vae=vae_s, self_token_critic=True).eval()
wp = torch.from_numpy(synth.normal("g8.to_pred.weight", (1, 128), 23)) * 0.2
bp = torch.from_numpy(synth.normal("g8.to_pred.bias", (1,), 23)) * 0.2
mg_self.token_critic.to_pred.weight.copy_(wp)
mg_self.token_critic.to_pred.bias.copy_(bp)
keys = sorted(k for k in mg_self.state_dict() if k.startswith("token_critic.") and not k.startswith("token_critic.net."))
assert keys == ["token_critic.to_pred.bias", "token_critic.to_pred.weight"], keys
assert "token_critic.net.to_logits.weight" in mg_self.state_dict()
images, ids = run_generate(mg_self, 8, 781)
save("gen_selfcritic_small", images=images, ids=ids, w_pred=wp, b_pred=bp)

# G9: can_remask_prev_masked=True (muse_maskgit_pytorch.py:609-612; requires no_mask_token_prob > 0)
mg_rm = MaskGit(image_size=16, transformer=tr, vae=vae_s, no_mask_token_prob=0.1).eval()
images, ids = run_generate(mg_rm, 8, 782, can_remask_prev_masked=True)
save("gen_remask_prev_small", images=images, ids=ids)

# ------------------------------------------------------------------ G10: Muse cascade (muse_maskgit_pytorch.py:745-791) on the G4 / G5 models
from muse_maskgit_pytorch import Muse                               # noqa: E402

tr.encode_text = lambda texts: te[:2]
tr2.encode_text = lambda texts: te[:2]
muse = Muse(base=mg, superres=mg2)
torch.manual_seed(783)
calls = []
orig = vae_s.decode_from_ids           # base.vae and superres.vae are both eval copies of vae_s: wrap each
wrapped = []
for m_ in (mg, mg2):
    o_ = m_.vae.decode_from_ids
    wrapped.append((m_.vae, o_))
    m_.vae.decode_from_ids = lambda ids_, _o=o_: (calls.append(ids_.clone()), _o(ids_))[1]
sup, low = muse(["a"] * 2, timesteps=6, superres_timesteps=8, return_lowres=True, return_pil_images=False)
for v_, o_ in wrapped:
    v_.decode_from_ids = o_
assert len(calls) == 2
save("muse_small", lowres=low, superres=sup, base_ids=calls[0], superres_ids=calls[1])

# ------------------------------------------------------------------ G11: checkpoints WRITTEN BY THE REFERENCE (save(): muse_maskgit_pytorch.py:482-489,
# vqgan_vae.py:405-420), default-initialised modules; the cond_vae of the super-res model is a full VQGanVAE (with its discriminator,
# whose tensors the reference saves under cond_vae.discr.*), and the cascade output those weights produce
seed_t5("synth-64", 64)
torch.manual_seed(900)
vae_ck = VQGanVAE(dim=16, layers=2, codebook_size=256)
vae_ck2 = VQGanVAE(dim=16, layers=2, codebook_size=256)
tr_b = MaskGitTransformer(num_tokens=256, dim=64, seq_len=16, depth=1, dim_head=64, heads=1, t5_name="synth-64", flash=False)
tr_s = MaskGitTransformer(num_tokens=256, dim=64, seq_len=64, depth=1, dim_head=64, heads=1, t5_name="synth-64", flash=False)
base_ck = MaskGit(image_size=16, transformer=tr_b, vae=vae_ck).eval()
sr_ck = MaskGit(image_size=32, transformer=tr_s, vae=vae_ck, cond_vae=vae_ck2, cond_image_size=16).eval()
vae_ck.eval().save(os.path.join(HERE, "ckpt_vae.pt"))
base_ck.save(os.path.join(HERE, "ckpt_base.pt"))
sr_ck.save(os.path.join(HERE, "ckpt_superres.pt"))
sd_sr = torch.load(os.path.join(HERE, "ckpt_superres.pt"))
assert any(k.startswith("cond_vae.discr.") for k in sd_sr) and any(k.startswith("discr.") for k in torch.load(os.path.join(HERE, "ckpt_vae.pt")))
te64 = text_embeds("g11.te", 2, 8, 64, 31)
tr_b.encode_text = lambda texts: te64
tr_s.encode_text = lambda texts: te64
muse_ck = Muse(base=base_ck, superres=sr_ck)
torch.manual_seed(901)
calls = []
wrapped = []
for m_ in (base_ck, sr_ck):
    o_ = m_.vae.decode_from_ids
    wrapped.append((m_.vae, o_))
    m_.vae.decode_from_ids = lambda ids_, _o=o_: (calls.append(ids_.clone()), _o(ids_))[1]
sup, low = muse_ck(["a"] * 2, timesteps=4, superres_timesteps=4, return_lowres=True, return_pil_images=False)
for v_, o_ in wrapped:
    v_.decode_from_ids = o_
img = torch.from_numpy(synth.uniform("g11.img", (2, 3, 16, 16), 31))
_, vids, _ = vae_ck.encode(img)
save("ckpt_muse", lowres=low, superres=sup, base_ids=calls[0], superres_ids=calls[1], vae_ids=vids.long(), vae_recon=vae_ck.decode_from_ids(vids))
print("done")

# ------------------------------------------------------------------ G12: VAE with a non-default encoder / decoder layout
# per-stage res-block counts (1, 2) and a 3x3 stem (vqgan_vae.py:185-232): the weights travel inside the fixture (default init under a seed)
torch.manual_seed(31)
vae_v = VQGanVAE(dim=16, layers=2, codebook_size=256, encdec_layer_mults=(2, 4), encdec_num_resnet_blocks=(1, 2), encdec_first_conv_kernel_size=3).eval()
img = torch.from_numpy(synth.uniform("g12.img", (2, 3, 16, 16), 31))
fq, ids, _ = vae_v.encode(img)
sd_v = {k: v for k, v in vae_v.state_dict().items() if not k.startswith(("discr.", "_vgg."))}
save("vae_variant", img=img, ids=ids.long(), recon=vae_v.decode_from_ids(ids), fmap=vae_v.enc_dec.encode(img),
     **{"sd." + k: v for k, v in sd_v.items()})
