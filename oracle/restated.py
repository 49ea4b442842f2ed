"""ORACLE — TEST INFRASTRUCTURE ONLY. Never imported by the product path (visrag_b200/); only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may call it.

CPU fp32 restatement of the VisRAG-Ret embedding + retrieval hot path, written from the reference sources
(paths relative to /root/reference; every function cites the lines it follows). The arithmetic is floating
point, so it is plain fp32 PyTorch-on-CPU / numpy (third-party primitives the reference itself calls:
``F.interpolate``, ``F.layer_norm``, ``erf``-GELU, ``softmax``, ``PIL.Image.resize``).

Pinning: the reference has NO tests or golden vectors for this path (SURVEY.md §4, F11). This oracle is
pinned against the reference *itself*, executed through ``oracle/reference_shim.py`` to produce
``tests/golden/reference_checks.npz`` (``tests/test_oracle_vs_reference.py``) and against the golden
vectors generated from the real reference by ``oracle/gen_golden.py`` (``tests/golden/*.npz``,
``tests/test_oracle_golden.py`` — runs everywhere).

Differences from the reference that do not change results for valid tokens: sequences are processed one at a
time instead of right-padded batches (padding rows carry weight 0 in the pooling, `dense_retrieval_model.py:181`),
and every slice goes through the ViT on its own (the reference batches slices 1..n of a page,
`modeling_minicpmv.py:119`).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F
from PIL import Image

SD = Dict[str, torch.Tensor]


# ----------------------------------------------------------------------------------------------------
# A.1 page geometry  (modeling_minicpmv/modeling_minicpmv.py:482-592)
# ----------------------------------------------------------------------------------------------------
def ensure_divide(length: float, patch_size: int) -> int:
    """`modeling_minicpmv.py:540-541`."""
    return max(round(length / patch_size) * patch_size, patch_size)


def find_best_resize(original_size, scale_resolution: int, patch_size: int, allow_upscale: bool = False):
    """`modeling_minicpmv.py:544-552`."""
    width, height = original_size
    if (width * height > scale_resolution * scale_resolution) or allow_upscale:
        r = width / height
        height = int(scale_resolution / math.sqrt(r))
        width = int(height * r)
    return (ensure_divide(width, patch_size), ensure_divide(height, patch_size))


def get_refine_size(original_size, grid, scale_resolution: int, patch_size: int, allow_upscale: bool = False):
    """`modeling_minicpmv.py:555-575`."""
    width, height = original_size
    gx, gy = grid
    refine_w = ensure_divide(width, gx)
    refine_h = ensure_divide(height, gy)
    best = find_best_resize((refine_w / gx, refine_h / gy), scale_resolution, patch_size, allow_upscale=allow_upscale)
    return (best[0] * gx, best[1] * gy)


def slice_image(image: Image.Image, max_slice_nums: int = 9, scale_resolution: int = 448, patch_size: int = 14):
    """`modeling_minicpmv.py:482-537`. Returns (source_image, patches[row][col], best_grid or None)."""
    W, H = image.size
    log_ratio = math.log(W / H)
    ratio = W * H / (scale_resolution * scale_resolution)
    multiple = min(math.ceil(ratio), max_slice_nums)
    patches: List[List[Image.Image]] = []
    best_grid = None
    if multiple <= 1:
        best = find_best_resize((W, H), scale_resolution, patch_size, allow_upscale=True)
        source = image.resize(best, Image.Resampling.BICUBIC)
    else:
        cands = [i for i in (multiple - 1, multiple, multiple + 1) if not (i == 1 or i > max_slice_nums)]
        best = find_best_resize((W, H), scale_resolution, patch_size)
        source = image.copy().resize(best, Image.Resampling.BICUBIC)
        grids = []
        for n in cands:
            m = 1
            while m <= n:
                if n % m == 0:
                    grids.append([m, n // m])
                m += 1
        best_grid, min_err = [1, 1], float("inf")
        for g in grids:
            err = abs(log_ratio - math.log(g[0] / g[1]))
            if err < min_err:
                best_grid, min_err = g, err
        refine = get_refine_size((W, H), best_grid, scale_resolution, patch_size, allow_upscale=True)
        refined = image.resize(refine, Image.Resampling.BICUBIC)
        # split_to_patches (`:578-592`): i over height, j over width
        rw, rh = refined.size
        cw, ch = int(rw / best_grid[0]), int(rh / best_grid[1])
        for i in range(0, rh, ch):
            row = []
            for j in range(0, rw, cw):
                row.append(refined.crop((j, i, j + cw, i + ch)))
            patches.append(row)
    return source, patches, best_grid


# ----------------------------------------------------------------------------------------------------
# A.1/A.2 context string + tokens  (modeling_visrag_ret.py:57-84; modeling_minicpmv.py:173-216,247-274,595-609)
# ----------------------------------------------------------------------------------------------------
def prepare_context(text: str, image: Optional[Image.Image], tokenizer, query_num: int = 64, max_slice_nums: int = 9,
                    scale_resolution: int = 448, patch_size: int = 14):
    """`modeling_visrag_ret.py:57-84` with slice_mode=True. Returns (content, [slice images in LM order])."""
    if not image:
        return text, []
    ph = tokenizer.im_start + tokenizer.unk_token * query_num + tokenizer.im_end
    source, patches, grid = slice_image(image, max_slice_nums, scale_resolution, patch_size)
    images = [source]
    final = ph
    if len(patches) > 0:
        for row in patches:
            images.extend(row)
        cols, rows = grid[0], grid[1]  # `modeling_minicpmv.py:600-601`
        lines = ["".join([ph] * cols) for _ in range(rows)]
        final += tokenizer.slice_start + "\n".join(lines) + tokenizer.slice_end
    return final + "\n" + text, images


def convert_to_tensors(tokenizer, content: str, max_inp_length: Optional[int]):
    """`modeling_minicpmv.py:173-200`: ids (int64 numpy) and image_bound [n,2] = (pos(<image>)+1, pos(</image>))."""
    ids = tokenizer.encode(content) if tokenizer.add_bos_token else [tokenizer.bos_id] + tokenizer.encode(content)
    if max_inp_length is not None:
        ids = ids[:max_inp_length]
    ids = np.asarray(ids, dtype=np.int64)
    starts = np.where(ids == tokenizer.im_start_id)[0] + 1
    ends = np.where(ids == tokenizer.im_end_id)[0]
    n = max(len(starts), len(ends))
    bound = np.stack([starts[:n], ends[:n]], axis=1) if n > 0 else np.zeros((0, 2), dtype=np.int64)
    return ids, bound


def pixel_values(img: Image.Image) -> torch.Tensor:
    """ToTensor + Normalize(0.5, 0.5) (`modeling_minicpmv.py:84-92`): fp32 CHW in [-1, 1]."""
    a = np.asarray(img.convert("RGB"), dtype=np.uint8)
    x = torch.from_numpy(a.copy()).permute(2, 0, 1).float() / 255.0
    return (x - 0.5) / 0.5


# ----------------------------------------------------------------------------------------------------
# A.4 SigLIP ViT  (timm: patch_embed.py:68-93, pos_embed.py:17-57, vision_transformer.py:86-107,165-168,682-692)
# ----------------------------------------------------------------------------------------------------
def resample_pos_embed(pos: torch.Tensor, gh: int, gw: int) -> torch.Tensor:
    """`timm/layers/pos_embed.py:17-57` with num_prefix_tokens=0: bicubic + antialias in fp32; identity when the
    grid equals the native square grid. pos [1, S*S, D] -> [gh*gw, D]."""
    S = int(math.sqrt(pos.shape[1]))
    if gh * gw == pos.shape[1] and gh == gw:
        return pos[0]
    D = pos.shape[-1]
    p = pos.float().reshape(1, S, S, D).permute(0, 3, 1, 2)
    p = F.interpolate(p, size=(gh, gw), mode="bicubic", antialias=True)
    return p.permute(0, 2, 3, 1).reshape(gh * gw, D)


def vit_forward(sd: SD, cfg, px: torch.Tensor) -> torch.Tensor:
    """One slice [3,h,w] (h,w multiples of 14) -> [N, D] after the final LayerNorm.
    `VisionTransformer.forward_features` (`vision_transformer.py:682-692`)."""
    P, D, nh = cfg.patch_size, cfg.vit_dim, cfg.vit_heads
    hd = D // nh
    x = F.conv2d(px[None], sd["vpm.patch_embed.proj.weight"], sd["vpm.patch_embed.proj.bias"], stride=P)
    _, _, gh, gw = x.shape
    x = x.permute(0, 2, 3, 1).reshape(gh * gw, D)  # NHWC -> [N, D] (`patch_embed.py:88-91`, `:600-609`)
    x = x + resample_pos_embed(sd["vpm.pos_embed"], gh, gw)
    N = x.shape[0]
    for i in range(cfg.vit_depth):
        p = f"vpm.blocks.{i}."
        h = F.layer_norm(x, (D,), sd[p + "norm1.weight"], sd[p + "norm1.bias"], cfg.ln_eps)
        qkv = F.linear(h, sd[p + "attn.qkv.weight"], sd[p + "attn.qkv.bias"]).reshape(N, 3, nh, hd).permute(1, 2, 0, 3)
        q, k, v = qkv[0], qkv[1], qkv[2]  # [nh, N, hd]  (`vision_transformer.py:88-89`)
        att = torch.softmax((q * hd ** -0.5) @ k.transpose(-2, -1), dim=-1)
        o = (att @ v).transpose(0, 1).reshape(N, D)
        x = x + F.linear(o, sd[p + "attn.proj.weight"], sd[p + "attn.proj.bias"])
        h = F.layer_norm(x, (D,), sd[p + "norm2.weight"], sd[p + "norm2.bias"], cfg.ln_eps)
        h = F.gelu(F.linear(h, sd[p + "mlp.fc1.weight"], sd[p + "mlp.fc1.bias"]))  # exact erf GELU (`mlp.py:41-49`)
        x = x + F.linear(h, sd[p + "mlp.fc2.weight"], sd[p + "mlp.fc2.bias"])
    return F.layer_norm(x, (D,), sd["vpm.norm.weight"], sd["vpm.norm.bias"], cfg.ln_eps)


# ----------------------------------------------------------------------------------------------------
# A.5 Resampler  (resampler.py:38-90,146-168)
# ----------------------------------------------------------------------------------------------------
def sincos_2d(embed_dim: int, gh: int, gw: int) -> np.ndarray:
    """`resampler.py:38-90`: grid = meshgrid(w, h); first half of the channels encodes grid[0] (w index)."""
    grid_h = np.arange(gh, dtype=np.float32)
    grid_w = np.arange(gw, dtype=np.float32)
    grid = np.stack(np.meshgrid(grid_w, grid_h), axis=0).reshape(2, 1, gh, gw)

    def one(dim, pos):
        omega = np.arange(dim // 2, dtype=np.float32)
        omega /= dim / 2.0
        omega = 1.0 / 10000 ** omega
        out = np.einsum("m,d->md", pos.reshape(-1), omega)
        return np.concatenate([np.sin(out), np.cos(out)], axis=1)

    return np.concatenate([one(embed_dim // 2, grid[0]), one(embed_dim // 2, grid[1])], axis=1)


def resampler_forward(sd: SD, cfg, x: torch.Tensor, gh: int, gw: int) -> torch.Tensor:
    """[N, D] -> [64, E]  (`Resampler.forward`, `resampler.py:146-168`; nn.MultiheadAttention math)."""
    E = cfg.hidden
    nh = E // 128
    pos = torch.from_numpy(sincos_2d(E, gh, gw)).float()
    kv = F.layer_norm(F.linear(x, sd["resampler.kv_proj.weight"]), (E,), sd["resampler.ln_kv.weight"],
                      sd["resampler.ln_kv.bias"], 1e-6)
    q_in = F.layer_norm(sd["resampler.query"], (E,), sd["resampler.ln_q.weight"], sd["resampler.ln_q.bias"], 1e-6) \
        + sd["resampler.pos_embed"]
    W, b = sd["resampler.attn.in_proj_weight"], sd["resampler.attn.in_proj_bias"]
    q = F.linear(q_in, W[:E], b[:E])
    k = F.linear(kv + pos, W[E:2 * E], b[E:2 * E])
    v = F.linear(kv, W[2 * E:], b[2 * E:])
    Q = q.reshape(-1, nh, 128).transpose(0, 1)
    K = k.reshape(-1, nh, 128).transpose(0, 1)
    V = v.reshape(-1, nh, 128).transpose(0, 1)
    att = torch.softmax((Q * 128 ** -0.5) @ K.transpose(-2, -1), dim=-1)
    o = (att @ V).transpose(0, 1).reshape(-1, E)
    o = F.linear(o, sd["resampler.attn.out_proj.weight"], sd["resampler.attn.out_proj.bias"])
    o = F.layer_norm(o, (E,), sd["resampler.ln_post.weight"], sd["resampler.ln_post.bias"], 1e-6)
    return o @ sd["resampler.proj"]


def vision_embedding(sd: SD, cfg, slices: Sequence[Image.Image]) -> torch.Tensor:
    """`get_vision_embedding` (`modeling_minicpmv.py:95-122`): all slices of one page -> [n*64, E]."""
    outs = []
    for im in slices:
        px = pixel_values(im)
        gh, gw = math.ceil(px.shape[1] / cfg.patch_size), math.ceil(px.shape[2] / cfg.patch_size)
        outs.append(resampler_forward(sd, cfg, vit_forward(sd, cfg, px), gh, gw))
    return torch.cat(outs, dim=0)


# ----------------------------------------------------------------------------------------------------
# A.6/A.7 MiniCPM decoder  (modeling_minicpm.py:119-123,142-182,259-290,333,824-910,939-1004,1147-1304)
# ----------------------------------------------------------------------------------------------------
def rms_norm(x: torch.Tensor, w: torch.Tensor, eps: float) -> torch.Tensor:
    """`modeling_minicpm.py:119-123`."""
    var = x.float().pow(2).mean(dim=-1, keepdim=True)
    return x * torch.rsqrt(var + eps) * w


def rope_tables(hd: int, theta: float, L: int):
    """`MiniCPMRotaryEmbedding` (`:142-182`): cos/sin of cat(freqs, freqs), fp32."""
    inv = 1.0 / (theta ** (torch.arange(0, hd, 2).float() / hd))
    fr = torch.outer(torch.arange(L).float(), inv)
    emb = torch.cat([fr, fr], dim=-1)
    return emb.cos(), emb.sin()


def lm_forward(sd: SD, cfg, h: torch.Tensor) -> torch.Tensor:
    """One unpadded sequence of input embeddings [L, H] -> final-norm hidden states [L, H]."""
    L, H = h.shape
    nh, hd = cfg.heads, cfg.hidden // cfg.heads
    cos, sin = rope_tables(hd, cfg.rope_theta, L)
    s = cfg.scale_depth / math.sqrt(cfg.layers)
    causal = torch.full((L, L), float("-inf")).triu(1)

    def rot(x):  # rotate_half (`:252-256`)
        return torch.cat([-x[..., hd // 2:], x[..., : hd // 2]], dim=-1)

    for i in range(cfg.layers):
        p = f"llm.model.layers.{i}."
        a = rms_norm(h, sd[p + "input_layernorm.weight"], cfg.rms_eps)
        q = F.linear(a, sd[p + "self_attn.q_proj.weight"]).reshape(L, nh, hd).transpose(0, 1)
        k = F.linear(a, sd[p + "self_attn.k_proj.weight"]).reshape(L, nh, hd).transpose(0, 1)
        v = F.linear(a, sd[p + "self_attn.v_proj.weight"]).reshape(L, nh, hd).transpose(0, 1)
        q = q * cos + rot(q) * sin
        k = k * cos + rot(k) * sin
        att = torch.softmax(q @ k.transpose(-2, -1) / math.sqrt(hd) + causal, dim=-1)
        o = (att @ v).transpose(0, 1).reshape(L, H)
        h = h + F.linear(o, sd[p + "self_attn.o_proj.weight"]) * s
        m = rms_norm(h, sd[p + "post_attention_layernorm.weight"], cfg.rms_eps)
        m = F.linear(F.silu(F.linear(m, sd[p + "mlp.gate_proj.weight"])) * F.linear(m, sd[p + "mlp.up_proj.weight"]),
                     sd[p + "mlp.down_proj.weight"])
        h = h + m * s
    return rms_norm(h, sd["llm.model.norm.weight"], cfg.rms_eps)


def lm_inputs(sd: SD, cfg, ids: np.ndarray, bound: np.ndarray, vis: Optional[torch.Tensor]) -> torch.Tensor:
    """`get_vllm_embedding` (`modeling_minicpmv.py:139-166`): embed*scale_emb, vision rows scattered into image_bound."""
    e = sd["llm.model.embed_tokens.weight"][torch.from_numpy(ids)] * cfg.scale_emb
    if vis is not None and len(bound) > 0:
        idx = torch.cat([torch.arange(int(r[0]), int(r[1])) for r in bound])
        e = e.clone()
        e[idx] = vis.reshape(-1, vis.shape[-1])[: len(idx)]
    return e


# ----------------------------------------------------------------------------------------------------
# A.8 pooling + normalise  (dense_retrieval_model.py:170-223)
# ----------------------------------------------------------------------------------------------------
def pool(hidden: torch.Tensor, pooling: str = "wmean") -> torch.Tensor:
    """Unpadded [L, H] -> [H]. wmean: w_t = t+1 (`dense_retrieval_model.py:180-184`)."""
    L = hidden.shape[0]
    if pooling == "wmean":
        w = torch.arange(1, L + 1, dtype=torch.float32)
        return (hidden * w[:, None]).sum(0) / w.sum()
    if pooling == "mean":
        return hidden.sum(0) / float(L)
    if pooling == "lasttoken":
        return hidden[-1]
    if pooling == "cls":
        return hidden[0]
    raise ValueError(pooling)


def encode(sd: SD, cfg, tokenizer, texts: List[str], images: List[Optional[Image.Image]], max_inp_length: int = 2048,
           pooling: str = "wmean", return_hidden: bool = False):
    """`DRModel.encode` over `VisRAG_Ret.forward` (`dense_retrieval_model.py:142-225`, `modeling_visrag_ret.py:86-126`).
    Returns fp32 numpy [B, H] (L2-normalised)."""
    reps, hiddens = [], []
    with torch.no_grad():
        for text, image in zip(texts, images):
            content, slices = prepare_context(text, image, tokenizer, cfg.query_num, cfg.max_slice_nums,
                                              cfg.scale_resolution, cfg.patch_size)
            ids, bound = convert_to_tensors(tokenizer, content, max_inp_length)
            vis = vision_embedding(sd, cfg, slices) if slices else None
            h = lm_forward(sd, cfg, lm_inputs(sd, cfg, ids, bound, vis))
            r = pool(h, pooling)
            reps.append(F.normalize(r[None], dim=1)[0])  # eps 1e-12 (`:222-223`)
            hiddens.append(h.numpy())
    out = torch.stack(reps).numpy().astype(np.float32)
    return (out, hiddens) if return_hidden else out


# ----------------------------------------------------------------------------------------------------
# A.9 score + top-k  (retriever/dense_retriever.py:25-30)
# ----------------------------------------------------------------------------------------------------
def score_topk(Q: np.ndarray, D: np.ndarray, k: int):
    """S = Q D^T in fp32, top-k largest per row, sorted descending (ties: lower index first).
    Returns (scores [nq,k] f32, indices [nq,k] i64)."""
    S = torch.from_numpy(np.ascontiguousarray(Q, dtype=np.float32)) @ torch.from_numpy(
        np.ascontiguousarray(D, dtype=np.float32)).T
    k = min(k, S.shape[1])
    # stable sort on (-score, index) gives a deterministic tie rule; torch.topk's is unspecified
    order = torch.sort(-S, dim=1, stable=True).indices[:, :k]
    return torch.gather(S, 1, order).numpy(), order.numpy().astype(np.int64)


def merge_topk(parts: List[Tuple[np.ndarray, np.ndarray]], k: int):
    """k-way merge of per-shard (scores, global ids): the union dict of `dense_retriever.py:88-92` re-truncated to k
    by (score desc, id asc)."""
    s = np.concatenate([p[0] for p in parts], axis=1)
    i = np.concatenate([p[1] for p in parts], axis=1)
    order = np.lexsort((i, -s), axis=1)[:, :k]
    return np.take_along_axis(s, order, 1), np.take_along_axis(i, order, 1)


def recall_at_k(run_ids: np.ndarray, relevant: List[set], k: int) -> float:
    """Recall@k = |top-k ∩ relevant| / |relevant| averaged over queries (pytrec_eval `recall.k` semantics,
    `driver/eval.py:281-283`)."""
    vals = []
    for q, rel in enumerate(relevant):
        if not rel:
            continue
        vals.append(len(set(int(x) for x in run_ids[q, :k]) & rel) / len(rel))
    return float(np.mean(vals)) if vals else 0.0
