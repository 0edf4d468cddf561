"""Deterministic RWKV-7 test weights (shared by make_rwkv7_golden.py and the tests, so the golden file only has to hold
token ids and expected logits).  Tensor names / shapes follow candle_rwkv7/convert_pth_direct.py:11-134 and the loader in
candle_rwkv7/src/models/rwkv7.rs:105-144, 404-409, 443-506.  Every value is bf16-exact, so the f32 oracle and the bf16
device weights are bit-identical."""
import numpy as np

RWKV7_TINY = dict(arch=1, vocab=320, d_model=128, n_layers=3, n_heads=2, n_kv_heads=0, head_dim=64, d_ffn=512, norm_eps=1e-5,
                  rope_theta=0.0, lora_w=64, lora_a=64, lora_v=32, lora_g=128)


def bf16_exact(a):
    a = np.ascontiguousarray(a, np.float32)
    u = a.view(np.uint32).astype(np.uint64)
    u = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return u.astype(np.uint32).view(np.float32)


def make_weights(cfg, seed=0):
    rng = np.random.default_rng(seed)
    C, F, V, L = cfg["d_model"], cfg["d_ffn"], cfg["vocab"], cfg["n_layers"]
    W = {}

    def lin(name, out, inp, scale=1.0):
        W[name] = rng.normal(0, scale / np.sqrt(inp), (out, inp))

    def vec(name, mean, std):
        W[name] = rng.normal(mean, std, C)

    W["model.embeddings.weight"] = rng.normal(0, 1.0, (V, C))
    for l in range(L):
        p = f"model.layers.{l}."
        if l == 0:
            vec(p + "pre_norm.weight", 1.0, 0.1)
            vec(p + "pre_norm.bias", 0.0, 0.1)
        for nm in ("attn_norm", "ffn_norm"):
            vec(p + nm + ".weight", 1.0, 0.1)
            vec(p + nm + ".bias", 0.0, 0.1)
        a = p + "attn."
        for nm in ("r_proj", "k_proj", "v_proj", "o_proj"):
            lin(a + nm + ".weight", C, C)
        vec(a + "g_norm.weight", 1.0, 0.1)
        vec(a + "g_norm.bias", 0.0, 0.1)
        for nm in ("x_r", "x_w", "x_k", "x_v", "x_a", "x_g"):
            W[a + nm] = rng.uniform(0.0, 1.0, C)
        vec(a + "k_k", 0.85, 0.1)
        vec(a + "k_a", 1.0, 0.1)
        vec(a + "r_k", 0.0, 0.3)
        lin(a + "w_lora.lora.0.weight", cfg["lora_w"], C)
        lin(a + "w_lora.lora.2.weight", C, cfg["lora_w"])
        vec(a + "w_lora.lora.2.bias", -1.0, 1.5)
        lin(a + "a_lora.lora.0.weight", cfg["lora_a"], C)
        lin(a + "a_lora.lora.2.weight", C, cfg["lora_a"])
        vec(a + "a_lora.lora.2.bias", 0.0, 1.0)
        if l > 0:
            lin(a + "v_lora.lora.0.weight", cfg["lora_v"], C)
            lin(a + "v_lora.lora.2.weight", C, cfg["lora_v"])
            vec(a + "v_lora.lora.2.bias", 0.0, 1.0)
        lin(a + "g_lora.lora.0.weight", cfg["lora_g"], C)
        lin(a + "g_lora.lora.2.weight", C, cfg["lora_g"], 2.0)
        W[p + "ffn.x_k"] = rng.uniform(0.0, 1.0, C)
        lin(p + "ffn.key.weight", F, C)
        lin(p + "ffn.value.weight", C, F)
    vec("model.norm.weight", 1.0, 0.1)
    vec("model.norm.bias", 0.0, 0.1)
    lin("lm_head.weight", V, C, 2.0)
    return {k: bf16_exact(v) for k, v in W.items()}


def long_memory(W, cfg, seed=1):
    """w_lora bias ~ N(-7, 0.5): decay ~ 0.999, the state keeps hundreds of tokens"""
    rng = np.random.default_rng(seed)
    W = dict(W)
    for l in range(cfg["n_layers"]):
        W[f"model.layers.{l}.attn.w_lora.lora.2.bias"] = bf16_exact(rng.normal(-7.0, 0.5, cfg["d_model"]))
    return W
