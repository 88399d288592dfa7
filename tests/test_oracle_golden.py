"""CPU: the oracle against fixtures produced by the REFERENCE's own code (tests/golden/make_golden.py,
tests/golden/make_golden_live.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import dbnet as odb
from oracle import parseq as ops
from oracle import pipeline as opipe
from oracle import weights

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# fp32 convolutions sum in an order that depends on the CPU's oneDNN kernels and the thread count: the prob maps of the
# fixtures' machine and another one differ by up to 1e-5 (4e-6 with 1-4 threads on the same machine)
DBNET_TOL = 3e-5


def test_dbnet_oracle_matches_reference_fixture():
    z = np.load(os.path.join(G, "dbnet_ref.npz"))
    sd = weights.make_dbnet_state_dict(seed=int(z["weight_seed"]))
    y = odb.dbnet_forward(sd, torch.from_numpy(z["x"]))
    assert y.shape == (1, 1, 64, 96)
    assert np.abs(y.numpy() - z["prob"]).max() < DBNET_TOL


@pytest.mark.parametrize("tag,kw", [("peaked", dict(peaked=True)), ("repeat", dict(peaked=True, degenerate_repeat=True)),
                                    ("random", dict())])
def test_parseq_oracle_matches_reference_fixture(tag, kw, charset_v2):
    z = np.load(os.path.join(G, "parseq_ref_%s.npz" % tag), allow_pickle=True)
    spec = ops.SPECS["parseq-tiny-dynw-v4"]
    sd = weights.make_parseq_state_dict(spec, seed=int(z["weight_seed"]), **kw)
    lg = ops.parseq_forward(sd, spec, torch.from_numpy(z["img"]))
    assert lg.shape == (3, 101, spec.num_classes)
    assert np.abs(lg[:, 0].numpy() - z["logits_pos0"]).max() < 5e-4
    assert np.array_equal(lg.argmax(-1).numpy(), z["ids"])
    strings, scores = ops.Tokenizer(charset_v2).decode(lg.softmax(-1))
    assert strings == list(z["strings"])
    assert np.allclose(scores, z["scores"], rtol=2e-3, atol=1e-30)
    if tag == "repeat":
        # the repetition stop must have fired: strings are one repeated unit long, not 100 tokens
        assert all(len(s) < 10 for s in strings)


def test_host_functions_match_reference_fixture():
    z = np.load(os.path.join(G, "host_ref.npz"))
    for (h, w), (rh, rw) in zip(z["sizes"], z["resized"]):
        assert opipe.detector_input_size(int(h), int(w)) == (int(rh), int(rw))
    page = z["page"]
    for i, q in enumerate(z["quads"].tolist()):
        for dyn, key in ((False, "fixed%d" % i), (True, "dyn%d" % i)):
            made = opipe.make_crop(page, q, (32, 800), dynamic_width=dyn)
            if int(z["valid%d" % i]) == 0:
                assert made is None
            else:
                assert np.array_equal(made[0], z[key])
    x = opipe.detector_preprocess(page[:, :, ::-1].copy(), shortest=1280, limit=1600)
    assert x.shape[1] == 3 and x.shape[2] % 32 == 0 and x.shape[3] % 32 == 0
    # standardisation arithmetic (reference standardization_image on a float image)
    std = z["std"]
    mine = ((page.astype(np.float32)[:, :, ::-1] / 255.0 - np.array((0.485, 0.456, 0.406))) /
            np.array((0.229, 0.224, 0.225))).astype(np.float32)
    assert np.array_equal(mine, std)


def test_repeat_detector_cases():
    f = ops.detect_repeat_onset
    assert f([1, 2, 3, 4]) is None
    assert f([5] * 8) == (0, 1)
    assert f([9, 5, 5, 5, 5, 5]) is None                 # 5 equal tokens: no period qualifies yet
    assert f([9, 5, 5, 5, 5, 5, 5, 5]) == (2, 2)         # ... but 6 of them are a period-2 unit repeated 3 times
    assert f([9] + [5] * 8) == (1, 1)
    assert f([7, 1, 2, 1, 2, 1, 2]) == (1, 2)              # period 2 repeated 3 times
    assert f([1, 2, 3, 1, 2, 3, 1, 2, 3]) == (0, 3)
    assert f([1, 2, 1, 2]) is None


def test_oracle_against_reference_modules_live(charset_v2):
    """The model cases of oracle/refcheck.py (`python -m oracle.refcheck` runs them against the reference modules
    themselves) against the reference's outputs stored by tests/golden/make_golden_live.py: DBNet prob map, PARSeq
    logits (argmax ids, per-row max / mean, a seeded sample) and tokenizer decode for eight decoder configurations, and
    the post-processing quads / scores of tests/golden/post_ref.npz."""
    import sys
    sys.path.insert(0, G)
    import make_golden_live as L
    from make_golden import POST_PARAMS
    z = np.load(os.path.join(G, "live_ref.npz"))
    o = odb.dbnet_forward(weights.make_dbnet_state_dict(seed=L.DBNET_WEIGHT_SEED), L.dbnet_input())
    assert np.abs(o.numpy() - z["dbnet_prob"]).max() < DBNET_TOL
    for k, (spec, sd, img) in enumerate(L.parseq_cases()):
        o = ops.parseq_forward(sd, spec, img)
        assert tuple(o.shape) == tuple(z["parseq%d_shape" % k]), k
        assert np.array_equal(o.argmax(-1).numpy(), z["parseq%d_ids" % k]), k
        assert np.abs(o.max(-1).values.numpy() - z["parseq%d_rowmax" % k]).max() < 2e-4, k
        assert np.abs(o.mean(-1).numpy() - z["parseq%d_rowmean" % k]).max() < 2e-4, k
        got = o.reshape(-1)[torch.from_numpy(L.sample_index(o.numel(), L.PARSEQ_SAMPLE, 100 + k))].numpy()
        assert np.abs(got - z["parseq%d_sample" % k]).max() < 2e-4, k
        strings, scores = ops.Tokenizer(charset_v2).decode(o.softmax(-1))
        assert strings == z["parseq%d_strings" % k].tolist(), k
        assert all(abs(a - b) <= 2e-3 * max(abs(b), 1e-30) for a, b in zip(scores, z["parseq%d_scores" % k])), k
    p = np.load(os.path.join(G, "post_ref.npz"))
    for name, kw in POST_PARAMS.items():
        for ci in range(2):
            q, s = opipe.dbnet_postprocess(p["prob%d" % ci].astype(np.float32) / 255.0,
                                           tuple(int(v) for v in p["ori%d" % ci]), **kw)
            assert q == p["%s_quads%d" % (name, ci)].tolist() and s == p["%s_scores%d" % (name, ci)].tolist()


def test_postprocessing_matches_reference_fixture():
    """Row R3: quads and scores the reference's own DBnetPostProcessor produced (tests/golden/post_ref.npz, generated by
    make_golden.py from /root/reference with the oracle's stand-ins for pyclipper / shapely) - the oracle AND the
    product's post-processor must reproduce them exactly: contour order, the max_candidates cut, size / score filters,
    minAreaRect corner order, scaling, rounding."""
    import sys
    sys.path.insert(0, G)
    from make_golden import POST_PARAMS
    from yomitoku_b200.postprocessor import DBnetPostProcessor
    z = np.load(os.path.join(G, "post_ref.npz"))
    checked = 0
    for name, kw in POST_PARAMS.items():
        for ci in range(2):
            prob = z["prob%d" % ci].astype(np.float32) / 255.0
            ori = tuple(int(v) for v in z["ori%d" % ci])
            rq, rs = z["%s_quads%d" % (name, ci)].tolist(), z["%s_scores%d" % (name, ci)].tolist()
            oq, os_ = opipe.dbnet_postprocess(prob, ori, **kw)
            pq, ps = DBnetPostProcessor(**kw)({"binary": prob[None, None]}, ori)
            assert oq == rq and pq == rq and len(rq) >= 10
            assert os_ == rs and ps == rs
            checked += len(rq)
    assert checked > 100


def test_vit_encoder_restatement_against_torch_transformer_layers():
    """The ViT encoder is the one model part whose defining code (timm 1.0.27 `VisionTransformer`) is not installable
    here; the oracle restates it (oracle/parseq.py: encoder_forward).  A timm `Block` without LayerScale / DropPath /
    qk-norm is the standard pre-LayerNorm transformer layer, so the restatement is compared with PyTorch's OWN
    implementation of that layer - `nn.TransformerEncoderLayer(norm_first=True, activation="gelu")` over
    `nn.MultiheadAttention` (packed q, k, v projection in timm's order, same head split and 1/sqrt(hd) scale) - fed
    with the same weights: an independent implementation, not a second copy of the restatement."""
    import torch.nn as nn
    from oracle import parseq as ops
    from oracle import weights
    spec = ops.SPECS["parseq-tiny-dynw-v4"]
    sd = weights.make_parseq_state_dict(spec, seed=5, peaked=True)
    D, heads, depth = spec.embed_dim, spec.enc_heads, spec.enc_depth
    layers = []
    for i in range(depth):
        p = "encoder.blocks.%d." % i
        hidden = sd[p + "mlp.fc1.weight"].shape[0]
        lyr = nn.TransformerEncoderLayer(D, heads, dim_feedforward=hidden, dropout=0.0, activation="gelu",
                                         layer_norm_eps=1e-6, batch_first=True, norm_first=True)
        with torch.no_grad():
            lyr.self_attn.in_proj_weight.copy_(sd[p + "attn.qkv.weight"])
            lyr.self_attn.in_proj_bias.copy_(sd[p + "attn.qkv.bias"])
            lyr.self_attn.out_proj.weight.copy_(sd[p + "attn.proj.weight"])
            lyr.self_attn.out_proj.bias.copy_(sd[p + "attn.proj.bias"])
            lyr.linear1.weight.copy_(sd[p + "mlp.fc1.weight"])
            lyr.linear1.bias.copy_(sd[p + "mlp.fc1.bias"])
            lyr.linear2.weight.copy_(sd[p + "mlp.fc2.weight"])
            lyr.linear2.bias.copy_(sd[p + "mlp.fc2.bias"])
            lyr.norm1.weight.copy_(sd[p + "norm1.weight"])
            lyr.norm1.bias.copy_(sd[p + "norm1.bias"])
            lyr.norm2.weight.copy_(sd[p + "norm2.weight"])
            lyr.norm2.bias.copy_(sd[p + "norm2.bias"])
        layers.append(lyr.eval())
    g = torch.Generator().manual_seed(0)
    images = torch.rand(3, 3, 32, 208, generator=g) * 2 - 1
    with torch.inference_mode():
        ref = ops.encoder_forward(sd, spec, images)
        # patch embedding + positional table as in the restatement, then PyTorch's layers, then the final LayerNorm
        x = torch.nn.functional.conv2d(images, sd["encoder.patch_embed.proj.weight"], sd["encoder.patch_embed.proj.bias"],
                                       stride=spec.patch)
        B, _, gh, gw = x.shape
        x = x.flatten(2).transpose(1, 2)
        fgh, fgw = spec.grid
        x = x + sd["encoder.pos_embed"].reshape(1, fgh, fgw, D)[:, :gh, :gw].reshape(1, gh * gw, D)
        for lyr in layers:
            x = lyr(x)
        got = torch.nn.functional.layer_norm(x, (D,), sd["encoder.norm.weight"], sd["encoder.norm.bias"], 1e-6)
    assert got.shape == ref.shape
    assert (got - ref).abs().max().item() < 2e-4 * max(1.0, ref.abs().max().item())
