"""GPU tests of features added after the rest of the GPU suite (the host logic they exercise also has CPU tests):

  * padded prompt batches in the Qwen2.5-VL prefill and left-padded batches in generate() (gpt_image_edit_b200/qwen2p5vl.py:
    padding_spans, _decoder(spans=))
  * VAE slicing (gpt_image_edit_b200/vae.py: enable_slicing), reached through FluxKontextPipeline.enable_vae_slicing
  * save_pretrained / from_pretrained of the Univa model (the key mapping itself round-trips on the CPU, test_qwen_host_cpu.py)
"""
import pytest
import torch

from test_qwen_gpu import IMG, VSTART, _models, _rel_l2

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]


@pytest.mark.parametrize("side", ["right", "left"])
def test_padded_batch_prefill(side):
    """A batch of prompts of different lengths (`processor(..., padding=True)`, train_denoiser.py batches > 1): every
    sequence attends to its own tokens only — checked on the real tokens against transformers given the same mask
    (right padding) and against this engine's own unpadded runs (both sides) — and a padding row gets a ZERO attention
    output in every layer, i.e. it only passes through the MLPs, as under transformers' flash_attention_2 path (the
    backend the reference selects): checked against that chain written out in fp32."""
    from gpt_image_edit_b200.qwen2p5vl import get_rope_index

    ref, mine = _models()
    g = torch.Generator().manual_seed(5)
    grid = torch.tensor([[1, 16, 8]])
    pix = torch.randn(128, 1176, generator=g).bfloat16()
    row_a = [1, 2, 3, VSTART] + [IMG] * 32 + [903] + list(range(10, 25))
    row_b = list(range(40, 51))
    n, nb, PAD = len(row_a), len(row_b), 7
    if side == "right":
        ids = torch.tensor([row_a, row_b + [PAD] * (n - nb)])
        mask = torch.tensor([[1] * n, [1] * nb + [0] * (n - nb)])
        real_b = slice(0, nb)
    else:
        ids = torch.tensor([row_a, [PAD] * (n - nb) + row_b])
        mask = torch.tensor([[1] * n, [0] * (n - nb) + [1] * nb])
        real_b = slice(n - nb, n)
    h = mine(ids.cuda(), pixel_values=pix.cuda(), attention_mask=mask.cuda(), image_grid_thw=grid)
    assert h.shape == (2, n, 256) and torch.isfinite(h.float()).all()
    # (1) the engine's own unpadded runs of the two prompts
    h_a = mine(torch.tensor([row_a]).cuda(), pixel_values=pix.cuda(), image_grid_thw=grid)
    h_b = mine(torch.tensor([row_b]).cuda())
    assert _rel_l2(h[0], h_a[0]) < 5e-3 and _rel_l2(h[1, real_b], h_b[0]) < 5e-3
    ref32 = ref.to("cuda", torch.float32)
    with torch.no_grad():
        for p in ref32.parameters():
            p.copy_(p.bfloat16().float())
        if side == "right":
            # (2) transformers with the same mask and the reference's position ids, real tokens only
            pos, _ = get_rope_index(ids, grid, mask, spatial_merge_size=2, image_token_id=IMG, vision_start_token_id=VSTART)
            h32 = ref32(input_ids=ids.cuda(), attention_mask=mask.cuda(), pixel_values=pix.cuda().float(),
                        image_grid_thw=grid.cuda(), position_ids=pos.cuda()).last_hidden_state
            assert _rel_l2(h[0], h32[0]) < 2e-2 and _rel_l2(h[1, real_b], h32[1, real_b]) < 2e-2
        # (3) padding rows: embedding -> (x += mlp(post_attention_layernorm(x))) per layer -> final norm
        lm = ref32.language_model
        x = lm.embed_tokens(torch.tensor([PAD], device="cuda"))
        for layer in lm.layers:
            x = x + layer.mlp(layer.post_attention_layernorm(x))
        want = lm.norm(x)[0]
    pad_rows = h[1][mask[1] == 0]
    assert pad_rows.shape[0] == n - nb
    assert all(_rel_l2(r, want) < 2e-2 for r in pad_rows)


def test_generate_takes_left_padded_batches_and_refuses_right_padded_ones():
    """KV-cache decode of a left-padded prompt batch: each row's forced-token logits equal those of the prompt decoded alone
    (the orchestration is checked against transformers' generate on the CPU, tests/test_qwen_decoder_host_cpu.py)."""
    from gpt_image_edit_b200 import _lib

    _, mine = _models()
    mine.W["lm_head"].copy_((torch.randn(mine.W["lm_head"].shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4))
                             * 0.2).bfloat16())
    a, b = list(range(10, 33)), [5, 6, 7, 40, 41, 42, 43]
    forced = torch.tensor([[11, 12, 13, 14], [21, 22, 23, 24]]).cuda()
    batch = torch.tensor([a, [0] * (len(a) - len(b)) + b]).cuda()
    mask = torch.tensor([[1] * len(a), [0] * (len(a) - len(b)) + [1] * len(b)]).cuda()
    _, sc = mine.generate(batch, attention_mask=mask, forced_tokens=forced, output_scores=True, eos_token_id=(999999,))
    _, sa = mine.generate(torch.tensor([a]).cuda(), forced_tokens=forced[:1], output_scores=True, eos_token_id=(999999,))
    _, sb = mine.generate(torch.tensor([b]).cuda(), forced_tokens=forced[1:], output_scores=True, eos_token_id=(999999,))
    got = torch.stack(sc, dim=1)
    assert _rel_l2(got[0], torch.stack(sa, dim=1)[0]) < 5e-3 and _rel_l2(got[1], torch.stack(sb, dim=1)[0]) < 5e-3
    with pytest.raises(_lib.B2FError, match="left-padded"):
        mine.generate(batch.flip(1), attention_mask=mask.flip(1), max_new_tokens=2)


def test_vae_slicing_runs_one_item_per_pass_with_the_same_results():
    """`pipe.enable_vae_slicing()` (reference flux_pipeline.py:615-630 -> AutoencoderKL.enable_slicing): one batch item per
    kernel sequence.  Every normalisation in the VAE is per item, so the outputs are those of the batched call."""
    from gpt_image_edit_b200 import _lib as L
    from gpt_image_edit_b200.pipeline import FluxKontextPipeline
    from gpt_image_edit_b200.vae import B200AutoencoderKL, VaeConfig

    vae = B200AutoencoderKL(VaeConfig(block_out_channels=(64, 128, 256, 256))).randomize_(seed=6)
    pipe = FluxKontextPipeline(transformer=None, vae=vae)
    g = torch.Generator(device="cuda").manual_seed(8)
    img = (torch.rand(3, 3, 64, 96, device="cuda", generator=g) * 2 - 1).bfloat16()
    z = torch.randn(3, 16, 8, 12, device="cuda", generator=g).bfloat16()
    want = vae.encode(img).latent_dist.mode(), vae.decode(z, return_dict=False)[0], vae.decode_u8(z)
    pipe.enable_vae_slicing()
    assert vae.use_slicing
    got = vae.encode(img).latent_dist.mode(), vae.decode(z, return_dict=False)[0], vae.decode_u8(z)
    pipe.disable_vae_slicing()
    assert not vae.use_slicing
    assert got[0].shape == want[0].shape and _rel_l2(got[0], want[0]) < 4e-3
    assert got[1].shape == want[1].shape and _rel_l2(got[1], want[1]) < 4e-3
    assert got[2].shape == want[2].shape and (got[2].int() - want[2].int()).abs().max().item() <= 1
    with pytest.raises(L.B2FError):
        pipe.enable_vae_tiling()


def test_univa_model_save_pretrained_from_pretrained_round_trip(tmp_path):
    """`model.save_pretrained(dir)` / `UnivaQwen2p5VLForConditionalGeneration.from_pretrained(dir, torch_dtype=bf16,
    attn_implementation="flash_attention_2")` (reference train_denoiser.py:492-494, cli.py:37-41): every tensor comes back under
    its checkpoint name and the reloaded model computes the same prompt embeddings."""
    from univa.models.qwen2p5vl.modeling_univa_qwen2p5vl import UnivaQwen2p5VLForConditionalGeneration
    from univa.serve import cli

    model, _, _ = cli.load_main_model_and_processor("", torch.device("cuda"), synthetic=True, small=True)
    model.save_pretrained(tmp_path / "univa")
    m2 = UnivaQwen2p5VLForConditionalGeneration.from_pretrained(str(tmp_path / "univa"), torch_dtype=torch.bfloat16,
                                                                attn_implementation="flash_attention_2")
    from gpt_image_edit_b200.checkpoint import univa_state_dict
    a, b = univa_state_dict(model), univa_state_dict(m2)
    assert set(a) == set(b) and "denoise_tower.denoiser.transformer_blocks.0.attn.to_q.weight" in a and "lm_head.weight" in a
    assert all(torch.equal(a[k], b[k]) for k in a)
    ids = cli.synthetic_chat_tokens(0).cuda()
    e1 = model(ids, attention_mask=torch.ones_like(ids), output_type="denoise_embeds")
    e2 = m2(ids, attention_mask=torch.ones_like(ids), output_type="denoise_embeds")
    assert torch.equal(e1, e2)
