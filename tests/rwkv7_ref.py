"""f64 restatement of RWKV-7 (TEST INFRASTRUCTURE): the same formulas as oracle/cz_rwkv7.c:96-202 (candle_rwkv7 rwkv7.rs
179-328, 412-430, 468-478, 509-524, 529-542), evaluated in float64 so that a CUDA kernel's f32 error can be measured against it.

The WKV state of a head is S[i][j]: row i follows the value index, column j the key index (rwkv7.rs:290-302).  The CUDA kernel
keeps it in HBM as S[(j/4)*64 + i] float4 over j%4 (csrc/rwkv7.cu), i.e. element (i, j) at (j/4)*256 + i*4 + j%4;
state_to_kernel / state_from_kernel restate that layout."""
import numpy as np

GN_EPS = 64e-5


def layer_norm(x, w, b, eps):
    """LayerNorm of every row of x (population variance, like candle's LayerNorm)"""
    x = np.asarray(x, np.float64)
    mean = x.mean(axis=-1, keepdims=True)
    c = x - mean
    var = (c * c).mean(axis=-1, keepdims=True)
    return c / np.sqrt(var + eps) * w + b


def token_shift_mix(xn, prev, mu):
    """xn + (prev - xn) * mu  (rwkv7.rs:191-201, 414-424)"""
    return xn + (prev - xn) * mu


def sigmoid(x):
    return 1.0 / (1.0 + np.exp(-x))


def decay(z):
    """w = exp(-exp(-softplus(-z) - 0.5)), softplus written as log(exp(-z) + 1) like the oracle and the kernel"""
    with np.errstate(over="ignore"):
        return np.exp(-np.exp(-np.log(np.exp(-z) + 1.0) - 0.5))


def state_to_kernel(S):
    """[..., H, 64 (i), 64 (j)] -> [..., H, 4096] in the kernel's layout"""
    S = np.asarray(S)
    return S.reshape(S.shape[:-2] + (64, 16, 4)).swapaxes(-3, -2).reshape(S.shape[:-2] + (4096,))


def state_from_kernel(K):
    K = np.asarray(K)
    return K.reshape(K.shape[:-1] + (16, 64, 4)).swapaxes(-3, -2).reshape(K.shape[:-1] + (64, 64))


def wkv7_step(S, r, k, v, wl, al, vl, g, vf, vecs, layer0):
    """One token of one stream: S [H][64][64] (updated in place), row inputs [C], vecs = dict of the eight per-channel vectors.
    Returns (out [C], v_first [C])."""
    H = S.shape[0]
    a = sigmoid(al + vecs["a0"])
    w = decay(wl + vecs["w0"])
    if layer0:
        vf = v
    else:
        v = v + (vf - v) * sigmoid(vl + vecs["v0"])
    kk = (k * vecs["k_k"]).reshape(H, 64)
    nrm = np.maximum(np.sqrt((kk * kk).sum(axis=1, keepdims=True)), 1e-12)
    kk = kk / nrm
    kt = k * (1.0 + (a - 1.0) * vecs["k_a"])
    w, a, kt, v, r = (q.reshape(H, 64) for q in (w, a, kt, v, r))
    sa = np.einsum("hij,hj->hi", S, kk)  # with the old state
    S *= w[:, None, :]
    S -= sa[:, :, None] * (kk * a)[:, None, :]
    S += v[:, :, None] * kt[:, None, :]
    y = np.einsum("hij,hj->hi", S, r)
    mean = y.mean(axis=1, keepdims=True)
    d = y - mean
    gn = d / np.sqrt((d * d).mean(axis=1, keepdims=True) + GN_EPS)
    alpha = (r * kt * vecs["r_k"].reshape(H, 64)).sum(axis=1, keepdims=True)
    out = ((gn * vecs["gn_w"].reshape(H, 64) + vecs["gn_b"].reshape(H, 64) + alpha * v) * g.reshape(H, 64)).reshape(-1)
    return out, vf


def wkv7_scan(S, rows, vf, vecs, layer0):
    """Consecutive rows of one stream: rows = dict r, k, v, wl, al, vl, g of [T][C]; vf [T][C].  S is updated in place.
    Returns (out [T][C], v_first [T][C])."""
    T = rows["r"].shape[0]
    out = np.empty((T, rows["r"].shape[1]))
    vf_out = np.array(vf, np.float64)
    for t in range(T):
        out[t], vf_out[t] = wkv7_step(S, *(rows[n][t] for n in ("r", "k", "v", "wl", "al", "vl", "g")), vf_out[t], vecs, layer0)
    return out, vf_out


def forward(cfg, W, tokens):
    """Logits [T][V] after each token of `tokens`, from a zero state: the whole f64 RWKV-7 forward, one layer at a time over the
    sequence (everything but the WKV scan is causal through the token shift alone)."""
    W = {n: np.asarray(a, np.float64) for n, a in W.items()}
    C, L, eps = cfg["d_model"], cfg["n_layers"], cfg["norm_eps"]
    H = C // 64
    T = len(tokens)

    def shift(xn):
        return np.vstack([np.zeros((1, C)), xn[:-1]])

    x = W["model.embeddings.weight"][np.asarray(tokens, np.int64)]
    vf = np.zeros((T, C))
    for l in range(L):
        p = f"model.layers.{l}."
        a = p + "attn."
        if l == 0:
            x = layer_norm(x, W[p + "pre_norm.weight"], W[p + "pre_norm.bias"], eps)
        xn = layer_norm(x, W[p + "attn_norm.weight"], W[p + "attn_norm.bias"], eps)
        prev = shift(xn)
        xr, xw, xk, xv, xa, xg = (token_shift_mix(xn, prev, W[a + q]) for q in ("x_r", "x_w", "x_k", "x_v", "x_a", "x_g"))
        rows = {
            "r": xr @ W[a + "r_proj.weight"].T,
            "k": xk @ W[a + "k_proj.weight"].T,
            "v": xv @ W[a + "v_proj.weight"].T,
            "wl": np.tanh(xw @ W[a + "w_lora.lora.0.weight"].T) @ W[a + "w_lora.lora.2.weight"].T,
            "al": (xa @ W[a + "a_lora.lora.0.weight"].T) @ W[a + "a_lora.lora.2.weight"].T,
            "vl": (xv @ W[a + "v_lora.lora.0.weight"].T) @ W[a + "v_lora.lora.2.weight"].T if l > 0 else np.zeros((T, C)),
            "g": sigmoid(xg @ W[a + "g_lora.lora.0.weight"].T) @ W[a + "g_lora.lora.2.weight"].T,
        }
        vecs = {"w0": W[a + "w_lora.lora.2.bias"], "a0": W[a + "a_lora.lora.2.bias"], "v0": W.get(a + "v_lora.lora.2.bias", np.zeros(C)),
                "k_k": W[a + "k_k"], "k_a": W[a + "k_a"], "r_k": W[a + "r_k"], "gn_w": W[a + "g_norm.weight"], "gn_b": W[a + "g_norm.bias"]}
        y, vf = wkv7_scan(np.zeros((H, 64, 64)), rows, vf, vecs, l == 0)
        x = x + y @ W[a + "o_proj.weight"].T
        xn = layer_norm(x, W[p + "ffn_norm.weight"], W[p + "ffn_norm.bias"], eps)
        xx = token_shift_mix(xn, shift(xn), W[p + "ffn.x_k"])
        x = x + np.maximum(xx @ W[p + "ffn.key.weight"].T, 0.0) ** 2 @ W[p + "ffn.value.weight"].T
    xn = layer_norm(x, W["model.norm.weight"], W["model.norm.bias"], eps)
    return xn @ W["lm_head.weight"].T
