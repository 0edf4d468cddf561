"""Host-side mirror of the reference's operator interface over the C ABI.

  Context            one GPU (one process per GPU)                       -> cz_init
  Model              SmolLmSession::load / Rwkv7Session::load            src/models.rs:48, 132
  Session            trait LanguageModelSession (batch-of-1 shim)        src/models.rs:28-33
  cdf_bounds/search  softmax_pdf + quantize_pdf_to_cdf (+ search)        src/main.rs:784-824, 2294-2299, 2622-2625
  ac_encode_lanes    ArithmeticEncoder::encode_counts + finish           src/main.rs:353-399
  Model.encode/decode  the coding loops + reprime schedule               src/main.rs:1979-2358, 2528-2653
  Model.xe_bits      cross_entropy_bits_over_span                        src/main.rs:1725-1751
Same names, argument meaning and error behaviour (errors raise CzError instead of anyhow::bail).
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import CzError, check, lib  # noqa: F401

_vp = C.c_void_p


def _f32(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a, a.ctypes.data_as(_lib.f32p)


def _u32(a):
    a = np.ascontiguousarray(a, dtype=np.uint32)
    return a, a.ctypes.data_as(_lib.u32p)


def _u64(a):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a, a.ctypes.data_as(_lib.u64p)


def _u8(a):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    return a, a.ctypes.data_as(_lib.u8p)


class Context:
    def __init__(self, device_id=0):
        h = _vp()
        check(lib.cz_init(device_id, C.byref(h)))
        self._h = h
        self.device_id = device_id

    def close(self):
        if self._h:
            lib.cz_shutdown(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def launch_count(self):
        return int(lib.cz_launch_count(self._h))

    def profile(self, mode=1):
        """0 off, 1 synchronous per-launch timing, 2 deferred event pairs (does not perturb a timed region)"""
        check(lib.cz_profile_enable(self._h, int(mode)))

    def stream_ptr(self):
        return int(lib.cz_ctx_stream(self._h) or 0)

    def profile_read(self, reset=True):
        nf = len(_lib.K_FAMILIES)
        ms = (C.c_double * nf)()
        n = (C.c_uint64 * nf)()
        check(lib.cz_profile_read(self._h, ms, n, 1 if reset else 0))
        out = {k: (ms[i], int(n[i])) for i, k in enumerate(_lib.K_FAMILIES)}
        g = [v for k, v in out.items() if k.startswith("gemm_")]
        out["gemm"] = (sum(x[0] for x in g), sum(x[1] for x in g))
        return out

    # ---- K1 ----
    def cdf_bounds(self, logits_vm, syms, mode=_lib.CZ_CDF_SMOLLM):
        """logits_vm: [V, M] vocab-major float32; syms: [M]. Returns (c_lo, c_hi) uint32 arrays."""
        a, p = _f32(logits_vm)
        v, m = a.shape
        s, sp = _u32(syms)
        lo = np.empty(m, np.uint32)
        hi = np.empty(m, np.uint32)
        check(lib.cz_cdf_bounds(self._h, p, v, m, m, mode, sp, lo.ctypes.data_as(_lib.u32p), hi.ctypes.data_as(_lib.u32p)))
        return lo, hi

    def cdf_search(self, logits_vm, values, mode=_lib.CZ_CDF_SMOLLM):
        a, p = _f32(logits_vm)
        v, m = a.shape
        s, sp = _u32(values)
        sym = np.empty(m, np.uint32)
        lo = np.empty(m, np.uint32)
        hi = np.empty(m, np.uint32)
        check(lib.cz_cdf_search(self._h, p, v, m, m, mode, sp, sym.ctypes.data_as(_lib.u32p), lo.ctypes.data_as(_lib.u32p),
                                hi.ctypes.data_as(_lib.u32p)))
        return sym, lo, hi

    def cdf_full(self, logits, mode=_lib.CZ_CDF_SMOLLM):
        a, p = _f32(logits)
        v = a.shape[0]
        n = (v + 256 if mode == _lib.CZ_CDF_RWKV_LITERALS else v) + 1
        cdf = np.empty(n, np.uint32)
        check(lib.cz_cdf_full(self._h, p, v, mode, cdf.ctypes.data_as(_lib.u32p)))
        return cdf

    def xe_bits_cols(self, logits_vm, syms, mode=_lib.CZ_CDF_SMOLLM):
        a, p = _f32(logits_vm)
        v, m = a.shape
        s, sp = _u32(syms)
        out = np.empty(m, np.float64)
        check(lib.cz_xe_bits_cols(self._h, p, v, m, m, mode, sp, out.ctypes.data_as(_lib.f64p)))
        return out

    def cdf_entropy(self, logits_vm, mode=_lib.CZ_CDF_SMOLLM):
        """logits_vm: [V, M] vocab-major float32.  Returns float64 [M]: the expected code length in bits of each column's quantised coding
        distribution, 2^-30 sum_s w_s (30 - log2 w_s) over the widths w_s of the CDF the coder uses in `mode` (cz_cdf_entropy)."""
        a, p = _f32(logits_vm)
        v, m = a.shape
        out = np.empty(m, np.float64)
        check(lib.cz_cdf_entropy(self._h, p, v, m, m, mode, out.ctypes.data_as(_lib.f64p)))
        return out

    # ---- K2 / K3 ----
    def ac_encode_lanes(self, c_lo, c_hi, lane_off):
        """Returns a list of payload bytes, one per lane."""
        lo, lop = _u32(c_lo)
        hi, hip = _u32(c_hi)
        off, offp = _u64(lane_off)
        n_lanes = off.shape[0] - 1
        out_off = np.array([4 * int(off[l]) + 8 * l for l in range(n_lanes + 1)], dtype=np.uint64)
        out = np.zeros(int(out_off[-1]) + 16, np.uint8)
        out_len = np.zeros(n_lanes, np.uint64)
        check(lib.cz_ac_encode_lanes(self._h, lop, hip, offp, n_lanes, out.ctypes.data_as(_lib.u8p), out_off.ctypes.data_as(_lib.u64p),
                                     out_len.ctypes.data_as(_lib.u64p)))
        return [out[int(out_off[l]) : int(out_off[l]) + int(out_len[l])].tobytes() for l in range(n_lanes)]

    def ac_decode_lanes(self, payloads, lane_off, cdf):
        off, offp = _u64(lane_off)
        n_lanes = off.shape[0] - 1
        pay_len = np.array([len(p) for p in payloads], dtype=np.uint64)
        pay_off = np.concatenate([[0], np.cumsum(pay_len)[:-1]]).astype(np.uint64)
        blob, blobp = _u8(np.frombuffer(b"".join(payloads) + b"\0", dtype=np.uint8))
        c, cp = _u32(cdf)
        syms = np.empty(int(off[-1]), np.uint32)
        check(lib.cz_ac_decode_lanes(self._h, blobp, pay_off.ctypes.data_as(_lib.u64p), pay_len.ctypes.data_as(_lib.u64p), offp, n_lanes,
                                     cp, c.shape[0] - 1, syms.ctypes.data_as(_lib.u32p)))
        return syms


SMOLLM_135M = dict(arch=0, vocab=49152, d_model=576, n_layers=30, n_heads=9, n_kv_heads=3, head_dim=64, d_ffn=1536,
                   norm_eps=1e-5, rope_theta=1e5)
# small same-architecture config for fast tests (shapes obey the kernels' constraints: d % 64, ffn % 96)
SMOLLM_TINY = dict(arch=0, vocab=1024, d_model=192, n_layers=2, n_heads=3, n_kv_heads=1, head_dim=64, d_ffn=576,
                   norm_eps=1e-5, rope_theta=1e5)


# rwkv7-g1-0.1b (candle_rwkv7/convert_pth_direct.py:177-188)
RWKV7_0P1B = dict(arch=1, vocab=65536, d_model=768, n_layers=12, n_heads=12, n_kv_heads=0, head_dim=64, d_ffn=3072, norm_eps=1e-5,
                  rope_theta=0.0, lora_w=64, lora_a=64, lora_v=32, lora_g=128)


def split_segments(n_tokens, n_segments):
    """Contiguous, non-increasing segment lengths (longest first), as the lock-step decoder needs."""
    n_segments = max(1, min(n_segments, max(1, n_tokens)))
    base, rem = divmod(n_tokens, n_segments)
    lens = [base + (1 if g < rem else 0) for g in range(n_segments)]
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)


class Model:
    def __init__(self, ctx: Context, cfg: dict, engine=_lib.CZ_ENGINE_TCGEN05):
        c = _lib.ModelConfig()
        for k, v in cfg.items():
            setattr(c, k, v)
        c.engine = engine
        h = _vp()
        check(lib.cz_model_create(ctx._h, C.byref(c), C.byref(h)))
        self._h = h
        self.ctx = ctx
        self.cfg = dict(cfg)
        self.engine = engine

    def close(self):
        if self._h:
            lib.cz_model_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def random_init(self, seed=0, std=0.02, embed_std=None):
        check(lib.cz_model_random_init(self._h, seed, std, std if embed_std is None else embed_std))
        return self

    def load_safetensors(self, paths):
        arr = (C.c_char_p * len(paths))(*[p.encode() for p in paths])
        check(lib.cz_model_load_safetensors(self._h, arr, len(paths)))
        return self

    def set_tensor(self, name, array):
        a, p = _f32(array)
        check(lib.cz_model_set_tensor(self._h, name.encode(), a.ctypes.data_as(_vp), _lib.CZ_DTYPE_F32, a.size))

    def tensor_names(self):
        out = []
        for i in range(lib.cz_model_tensor_count(self._h)):
            nm = C.c_char_p()
            n = C.c_size_t()
            check(lib.cz_model_tensor_info(self._h, i, C.byref(nm), C.byref(n)))
            out.append((nm.value.decode(), n.value))
        return out

    def get_tensor(self, name, n):
        out = np.empty(n, np.float32)
        check(lib.cz_model_get_tensor(self._h, name.encode(), out.ctypes.data_as(_lib.f32p), n))
        return out

    def tensors(self):
        """All weights as float32 (exactly the bf16 values the kernels use) -- what tests hand to the oracle."""
        return {nm: self.get_tensor(nm, n) for nm, n in self.tensor_names()}

    def session(self):
        return Session(self)

    def watch_digests(self, n_tokens):
        """f-4: BLAKE3-128 of every coded token's logits vector (blake3_f32_bin16, src/main.rs:955-961), computed on the GPU by the
        next encode / decode calls.  Returns the uint8 array [n_tokens][16] they fill; watch_digests(0) switches it off."""
        if not n_tokens:
            check(lib.cz_model_set_digest_out(self._h, None, 0))
            self._digests = None
            return None
        self._digests = np.zeros((n_tokens, 16), np.uint8)
        check(lib.cz_model_set_digest_out(self._h, self._digests.ctypes.data_as(_lib.u8p), n_tokens))
        return self._digests

    def _schedule(self, n_tokens, seg_start, bos, context, reprime_interval, events, max_batch_tokens):
        s = _lib.Schedule()
        seg, segp = _u64(seg_start)
        s.context, s.reprime_interval = context, reprime_interval
        s.n_segments = seg.shape[0] - 1
        s.seg_start = segp
        s.bos = bos
        s.max_batch_tokens = max_batch_tokens
        keep = [seg]
        if events:
            arr = (_lib.PrimeEvent * len(events))()
            for k, ev in enumerate(events):  # (i, explicit prime tokens, hold_until[, hist_take])
                i, prime, hold = ev[:3]
                a, p = _u32(prime)
                keep.append(a)
                arr[k] = _lib.PrimeEvent(i, p, a.shape[0], hold, ev[3] if len(ev) > 3 else 0)
            s.events = arr
            s.n_events = len(events)
            keep.append(arr)
        return s, keep

    def set_pdf_floor(self, enabled):
        """code SmolLM streams with the floored pdf (CZ_CDF_SMOLLM_FLOOR) in the following encode / decode calls; RWKV-7 refuses"""
        check(lib.cz_model_set_pdf_floor(self._h, 1 if enabled else 0))

    def set_dictionary(self, symbols):
        """code every segment of the following encode / decode calls as if it followed `symbols` (cz_model_set_dictionary); None or an
        empty list clears it"""
        if symbols is None or len(symbols) == 0:
            check(lib.cz_model_set_dictionary(self._h, None, 0))
            return
        a, p = _u32(symbols)
        check(lib.cz_model_set_dictionary(self._h, p, a.shape[0]))

    def set_match(self, order):
        """code the following encode / decode calls with the match model of order `order` (1..16; 0 is off): cz_model_set_match"""
        check(lib.cz_model_set_match(self._h, int(order)))

    def watch_match(self, n_tokens):
        """The match model's per-token report (cz_model_set_match_out): returns (pred, w), uint32 arrays [n_tokens] that the next encode /
        decode calls with the match model on fill with each coded token's prediction (_lib.MATCH_NONE if none) and flag weight W (0 if
        none); watch_match(0) switches it off."""
        if not n_tokens:
            check(lib.cz_model_set_match_out(self._h, None, None, 0))
            self._match_out = None
            return None
        self._match_out = (np.zeros(n_tokens, np.uint32), np.zeros(n_tokens, np.uint32))
        check(lib.cz_model_set_match_out(self._h, self._match_out[0].ctypes.data_as(_lib.u32p), self._match_out[1].ctypes.data_as(_lib.u32p),
                                         n_tokens))
        return self._match_out

    def _with_dictionary(self, dictionary, call):
        """call() with the dictionary set, cleared again afterwards (no dictionary: nothing is set)"""
        if dictionary is None:
            return call()
        self.set_dictionary(dictionary)
        try:
            return call()
        finally:
            self.set_dictionary(None)

    def encode(self, ids, n_segments=1, bos=0, context=512, reprime_interval=512, events=None, seg_start=None, max_batch_tokens=0,
               pdf_floor=False, zero_width_out=False, dictionary=None, match_order=0):
        """ids: coded tokens (no BOS). Returns (list of per-segment payload bytes, seg_start).
        pdf_floor: code with softmax_pdf_floor (no token is zero-width); the stream must be decoded with pdf_floor=True too.
        zero_width_out: a zero-width token does not raise CZ_ERR_ZERO_WIDTH; returns (payloads, seg_start, first_zw) instead, first_zw
        a uint64 array with each segment's segment-relative index of its first zero-width token or _lib.NO_ZERO_WIDTH (a segment with
        an index has an unspecified payload: cz_model_set_zero_width_out).
        dictionary: symbols every segment is coded as if it followed (cz_model_set_dictionary); decode with the same ones.
        match_order: the match model's order K (1..16; 0 is off: cz_model_set_match); decode with the same order."""
        self.set_pdf_floor(pdf_floor)
        self.set_match(match_order)
        a, p = _u32(ids)
        n = a.shape[0]
        seg_start = split_segments(n, n_segments) if seg_start is None else np.asarray(seg_start, np.uint64)
        s, keep = self._schedule(n, seg_start, bos, context, reprime_interval, events, max_batch_tokens)
        cap = (8 if match_order else 4) * n + 8 * int(s.n_segments) + 16  # (a token codes a flag and a model interval at most)
        data = np.empty(cap, np.uint8)
        seg_off = np.zeros(int(s.n_segments) + 1, np.uint64)
        bs = _lib.Bitstreams(data.ctypes.data_as(_lib.u8p), cap, seg_off.ctypes.data_as(_lib.u64p))
        run = lambda: check(lib.cz_encode(self._h, p, n, C.byref(s), C.byref(bs)))  # noqa: E731
        if not zero_width_out:
            self._with_dictionary(dictionary, run)
        else:
            first_zw = np.zeros(max(1, int(s.n_segments)), np.uint64)
            check(lib.cz_model_set_zero_width_out(self._h, first_zw.ctypes.data_as(_lib.u64p), first_zw.shape[0]))
            try:
                self._with_dictionary(dictionary, run)
            finally:
                check(lib.cz_model_set_zero_width_out(self._h, None, 0))
        pay = [data[int(seg_off[g]) : int(seg_off[g + 1])].tobytes() for g in range(int(s.n_segments))]
        return (pay, seg_start, first_zw[: int(s.n_segments)]) if zero_width_out else (pay, seg_start)

    def analyze(self, ids, n_segments=1, seg_start=None, bos=0, context=512, reprime_interval=512, pdf_floor=False, max_batch_tokens=0,
                dictionary=None):
        """Where the bits go: encodes ids as encode() does, with the code-length and zero-width sinks set (cleared again afterwards).
        Returns a dict with
          payloads, seg_start   as encode() returns them
          first_zw              per segment, its first zero-width token (segment-relative) or _lib.NO_ZERO_WIDTH (that segment's
                                payload is unspecified)
          c_lo, c_hi            uint32 [n]: the interval each token was coded with
          bits                  float64 [n]: 30 - log2(c_hi - c_lo), the token's exact code length before coder overhead; +inf where the
                                interval is empty (a zero-width token)
          entropy               float64 [n]: the expected code length of the distribution the token was coded from (cz_cdf_entropy), in
                                the alphabet of the call (pdf_floor applies)
        dictionary as in encode()."""
        a, p = _u32(ids)
        n = a.shape[0]
        if self.cfg.get("arch", 0) == _lib.CZ_ARCH_RWKV7 and pdf_floor:
            raise ValueError("pdf_floor: RWKV-7 codes with a floored alphabet already")
        if context < 1 or reprime_interval < 1:
            raise ValueError("context and reprime_interval must be >= 1")
        if seg_start is None:
            if n_segments < 1:
                raise ValueError("n_segments must be >= 1")
            seg_start = split_segments(n, n_segments)
        else:
            seg_start = np.asarray(seg_start, np.uint64)
            if seg_start.ndim != 1 or seg_start.shape[0] < 2 or int(seg_start[0]) != 0 or int(seg_start[-1]) != n or np.any(np.diff(seg_start.astype(np.int64)) < 0):
                raise ValueError(f"seg_start must run from 0 to len(ids) = {n}, non-decreasing")
        self.set_pdf_floor(pdf_floor)
        self.set_match(0)  # analyze codes without the match model
        s, keep = self._schedule(n, seg_start, bos, context, reprime_interval, None, max_batch_tokens)
        n_seg = int(s.n_segments)
        cap = 4 * n + 8 * n_seg + 16
        data = np.empty(cap, np.uint8)
        seg_off = np.zeros(n_seg + 1, np.uint64)
        bs = _lib.Bitstreams(data.ctypes.data_as(_lib.u8p), cap, seg_off.ctypes.data_as(_lib.u64p))
        c_lo, c_hi, ent = np.zeros(max(n, 1), np.uint32), np.zeros(max(n, 1), np.uint32), np.zeros(max(n, 1), np.float64)
        first_zw = np.zeros(max(1, n_seg), np.uint64)
        check(lib.cz_model_set_zero_width_out(self._h, first_zw.ctypes.data_as(_lib.u64p), first_zw.shape[0]))
        try:
            check(lib.cz_model_set_code_length_out(self._h, c_lo.ctypes.data_as(_lib.u32p), c_hi.ctypes.data_as(_lib.u32p),
                                                   ent.ctypes.data_as(_lib.f64p), c_lo.shape[0]))
            self._with_dictionary(dictionary, lambda: check(lib.cz_encode(self._h, p, n, C.byref(s), C.byref(bs))))
        finally:
            check(lib.cz_model_set_code_length_out(self._h, None, None, None, 0))
            check(lib.cz_model_set_zero_width_out(self._h, None, 0))
        pay = [data[int(seg_off[g]) : int(seg_off[g + 1])].tobytes() for g in range(n_seg)]
        c_lo, c_hi, ent = c_lo[:n], c_hi[:n], ent[:n]
        return dict(payloads=pay, seg_start=seg_start, first_zw=first_zw[:n_seg], c_lo=c_lo, c_hi=c_hi, bits=code_length_bits(c_lo, c_hi),
                    entropy=ent)

    def decode(self, payloads, seg_start, bos=0, context=512, reprime_interval=512, max_batch_tokens=0, events=None, pdf_floor=False,
               dictionary=None, match_order=0):
        """events: the same gated hint primes the encoder was given (src/main.rs:2586-2614), single segment only;
        pdf_floor, dictionary, match_order: the settings the stream was encoded with"""
        self.set_pdf_floor(pdf_floor)
        self.set_match(match_order)
        seg_start = np.asarray(seg_start, np.uint64)
        n = int(seg_start[-1])
        s, keep = self._schedule(n, seg_start, bos, context, reprime_interval, events, max_batch_tokens)
        lens = np.array([len(p) for p in payloads], dtype=np.uint64)
        seg_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
        blob, blobp = _u8(np.frombuffer(b"".join(payloads) + b"\0", dtype=np.uint8))
        out = np.empty(max(n, 1), np.uint32)
        self._with_dictionary(dictionary, lambda: check(lib.cz_decode(self._h, blobp, seg_off.ctypes.data_as(_lib.u64p), n, C.byref(s),
                                                                      out.ctypes.data_as(_lib.u32p))))
        return out[:n]

    def xe_bits(self, jobs):
        """jobs: list of (prime_tokens, target_tokens). Returns float64 bits per job."""
        arr = (_lib.XeJob * len(jobs))()
        keep = []
        for k, (prime, targets) in enumerate(jobs):
            a, ap = _u32(prime)
            t, tp = _u32(targets)
            keep += [a, t]
            arr[k] = _lib.XeJob(ap, a.shape[0], tp, t.shape[0])
        out = np.zeros(len(jobs), np.float64)
        check(lib.cz_xe_bits(self._h, arr, len(jobs), out.ctypes.data_as(_lib.f64p)))
        return out

    def chunk_logits(self, prime, targets):
        a, ap = _u32(prime)
        t, tp = _u32(targets)
        out = np.empty((t.shape[0], self.cfg["vocab"]), np.float32)
        check(lib.cz_chunk_logits(self._h, ap, a.shape[0], tp, t.shape[0], out.ctypes.data_as(_lib.f32p)))
        return out


def xe_make_prime(history, hint, max_ctx=511):
    """prime = tail(history, max_ctx - |hint|) ++ hint[..max_ctx]   (src/main.rs:1727-1739)."""
    hint = np.asarray([] if hint is None else hint, np.uint32)
    history = np.asarray(history, np.uint32)
    hb = min(len(hint), max_ctx)
    take = min(max_ctx - hb, len(history))
    return np.concatenate([history[len(history) - take :], hint[:hb]]).astype(np.uint32)


def code_length_bits(c_lo, c_hi):
    """30 - log2(c_hi - c_lo) per interval of total 2^30 (float64), +inf for an empty interval"""
    w = np.asarray(c_hi, np.int64) - np.asarray(c_lo, np.int64)
    with np.errstate(divide="ignore"):
        return 30.0 - np.log2(w.astype(np.float64))


class Session:
    """trait LanguageModelSession (src/models.rs:28-33) for one stream; logits come back to the host like to_vec1()."""

    def __init__(self, model: Model):
        h = _vp()
        check(lib.cz_session_new(model._h, C.byref(h)))
        self._h = h
        self.model = model

    def vocab_size(self):
        return int(lib.cz_session_vocab_size(self._h))

    def max_context_length(self):
        return int(lib.cz_session_max_context_length(self._h))

    def index_pos(self):
        return int(lib.cz_session_index_pos(self._h))

    def step_logits_tensor(self, token_id):
        out = np.empty(self.vocab_size(), np.float32)
        check(lib.cz_session_step_logits(self._h, int(token_id), out.ctypes.data_as(_lib.f32p)))
        return out

    def reprime_with_history_and_get_last_logits_tensor(self, history):
        a, p = _u32(history)
        out = np.empty(self.vocab_size(), np.float32)
        check(lib.cz_session_reprime(self._h, p, a.shape[0], out.ctypes.data_as(_lib.f32p)))
        return out

    def close(self):
        if self._h:
            lib.cz_session_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
