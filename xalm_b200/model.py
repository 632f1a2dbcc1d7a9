"""Host-side mirror of the reference's operator surface for the forward path, over the C ABI.

Same names and call shapes as /root/reference/src/model.h so the parity tests read like the reference's own
call sites (main.cpp:44-128):

    xalm  = Xalm.load(path)                           # xalm.h:90
    model = Model.from_xalm(xalm, context)            # model.cpp:48
    state = InferenceState(model.config)              # model.h:96
    model.cuda(); state.cuda()                        # the two lines main.cpp:211-212 has commented out
    model.forward(state, token, pos, mode)            # model.h:272
    sampler.sample_argmax(state)                      # sampler.cpp:19

The compute is entirely in libxalm_cuda.so; a Model that has not been moved to the device cannot run
(the reference's CPU path is not reimplemented here — the `oracle/` restatement is test infrastructure only).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi
from . import types as T
from . import xalm_file as X

KV_SINKS = 2  # model.h:10


class InferenceMode:
    HYDRATE_KV_CACHE = capi.HYDRATE_KV_CACHE
    OUTPUT_LOGITS = capi.OUTPUT_LOGITS


class Xalm:
    @staticmethod
    def load(path: str) -> X.XalmFile:
        return X.XalmFile(path)


class InferenceState:
    """model.h:96-156.  After state.cuda() the scratch lives on the device; logits() is the pinned host buffer the
    backend copies into."""

    def __init__(self, config: dict):
        self.config = config
        self._logits = np.zeros(config["vocab_size"], dtype=np.float32)
        self._on_device = False

    def cuda(self):
        self._on_device = True
        return self

    def logits(self) -> np.ndarray:
        return self._logits


class Model:
    def __init__(self, config: dict, tensors: "dict[str, tuple[T.XType, tuple, np.ndarray]]"):
        """tensors: name -> (type, element shape, raw payload as a uint8 array)."""
        self.config = config
        self.tensors = tensors
        self._h = None
        self.tp_rank, self.tp_size = 0, 1

    # ---- Model::from_xalm (model.cpp:48-118) -------------------------------------------------------------
    @staticmethod
    def from_xalm(xalm: X.XalmFile, context: int = 0) -> "Model":
        config = X.parse_config(xalm.metadata, context)
        tensors = {}
        for name, shape in X.expected_tensors(config).items():
            if name not in xalm.tensors:
                raise KeyError(name)                                   # std::map::at in model.cpp:63
            ti = xalm.tensors[name]
            if tuple(ti.shape) != tuple(shape):
                raise ValueError(f"shape mismatch for {name}: {list(ti.shape)} vs {list(shape)} expected!")  # model.cpp:66-75
            tensors[name] = (ti.type, tuple(shape), xalm.raw(name))
        return Model(config, tensors)

    @staticmethod
    def from_tensors(config: dict, it) -> "Model":
        """Build from an iterator of (name, XType, array) such as synth.iter_tensors (no file involved)."""
        tensors = {}
        shapes = X.expected_tensors(config)
        for name, t, arr in it:
            if name in shapes:
                tensors[name] = (t, tuple(shapes[name]), np.ascontiguousarray(arr).view(np.uint8).reshape(-1))
        return Model(config, tensors)

    # ---- model.cuda() -----------------------------------------------------------------------------------------
    def cuda(self, device: int = 0, tp_rank: int = 0, tp_size: int = 1, comm_id: bytes | None = None, stream: int | None = None,
             release_host: bool = False, ipc_exchange=None, max_seqs: int = 1) -> "Model":
        """max_seqs > 1: a batched handle with that many sequence slots (forward_batch*, select_seq)."""
        L = capi.lib()
        h = C.c_void_p()
        cfg = capi.XalmConfig.from_dict(self.config)
        capi.check(L.xalm_cuda_create(C.byref(cfg), device, tp_rank, tp_size, C.byref(h)))
        self._h = h
        self.tp_rank, self.tp_size = tp_rank, tp_size
        self.max_seqs = max_seqs
        try:
            if max_seqs != 1:
                capi.check(L.xalm_cuda_set_batch(h, max_seqs))
            if stream is not None:
                capi.check(L.xalm_cuda_set_stream(h, C.c_void_p(stream)))
            if tp_size > 1:
                if comm_id is None or len(comm_id) != 128:
                    raise ValueError("tensor parallel needs the 128-byte communicator id from comm_unique_id()")
                buf = (C.c_char * 128).from_buffer_copy(comm_id)
                capi.check(L.xalm_cuda_comm_init(h, buf))
                if ipc_exchange is not None:
                    # peer-memory allreduce: export my buffer, let the host gather everyone's handle, import the table
                    mine = (C.c_char * 64)()
                    capi.check(L.xalm_cuda_ipc_export(h, mine))
                    table = ipc_exchange(bytes(mine))
                    if len(table) != 64 * tp_size:
                        raise ValueError("ipc_exchange must return tp_size x 64 bytes")
                    tb = (C.c_char * len(table)).from_buffer_copy(table)
                    capi.check(L.xalm_cuda_ipc_import(h, tb))
            for name in list(self.tensors.keys()):
                t, shape, raw = self.tensors[name]
                self.upload(name, t, shape, raw)
                if release_host:
                    del self.tensors[name]
            capi.check(L.xalm_cuda_finalize(h))
        except Exception:
            self.close()
            raise
        return self

    def upload(self, name: str, t: T.XType, shape, raw: np.ndarray):
        raw = np.ascontiguousarray(raw)
        shp = (C.c_int * len(shape))(*shape)
        capi.check(capi.lib().xalm_cuda_upload_tensor(self._h, name.encode(), t.id, shp, len(shape), raw.ctypes.data_as(C.c_void_p),
                                                      raw.nbytes))

    def shard_range(self, name: str) -> tuple:
        """(row0, row1, col0, col1) of the element shape this tensor-parallel rank keeps of tensor `name`."""
        r = (C.c_int * 4)()
        capi.check(capi.lib().xalm_cuda_shard_range(self._h, name.encode(), r))
        return tuple(r)

    def upload_shard(self, name: str, t: T.XType, shape, rng: tuple, raw: np.ndarray):
        """Upload only the block `rng` = shard_range(name) of a tensor whose full element shape is `shape`."""
        raw = np.ascontiguousarray(raw)
        shp = (C.c_int * len(shape))(*shape)
        r4 = (C.c_int * 4)(*rng)
        capi.check(capi.lib().xalm_cuda_upload_tensor_shard(self._h, name.encode(), t.id, shp, len(shape), r4, raw.ctypes.data_as(C.c_void_p),
                                                            raw.nbytes))

    @staticmethod
    def comm_unique_id() -> bytes:
        buf = (C.c_char * 128)()
        capi.check(capi.lib().xalm_cuda_comm_unique_id(buf))
        return bytes(buf)

    # ---- Model::forward (model.h:272) ------------------------------------------------------------------------
    def forward(self, state: InferenceState, token: int, pos: int, mode: int = InferenceMode.OUTPUT_LOGITS) -> None:
        if self._h is None:
            raise RuntimeError("Model.forward: the model is not on a CUDA device (call model.cuda()); this backend has no CPU path")
        lg = state.logits()
        capi.check(capi.lib().xalm_cuda_forward(self._h, token, pos, mode, lg.ctypes.data_as(C.c_void_p)
                                                if mode == InferenceMode.OUTPUT_LOGITS else None))

    def forward_argmax(self, token: int, pos: int) -> int:
        """forward + Sampler.sample_argmax with the sampler on the device (4 bytes back instead of the logits)."""
        out = C.c_int(0)
        capi.check(capi.lib().xalm_cuda_forward_argmax(self._h, token, pos, C.byref(out)))
        return out.value

    GREEDY_MAX_IN, GREEDY_MAX_OUT = 8, 16   # xalm_cuda_forward_greedy's limits on n_in and n_out

    def forward_greedy(self, tokens, pos: int, n_out: int) -> list:
        """tokens[0..n-2] hydrate positions pos..pos+n-2, tokens[-1] decodes at pos+n-1, then n_out - 1 more greedy steps each
        feed the previous step's token: the n_out greedy tokens, with one host synchronisation (the tokens never leave the
        device in between).  The cache and the logits left on the device are those of the equivalent forward / forward_argmax
        loop.  1 <= len(tokens) <= 8, 1 <= n_out <= 16."""
        tok = np.ascontiguousarray(tokens, dtype=np.int32).reshape(-1)
        if not 1 <= tok.size <= self.GREEDY_MAX_IN:
            raise ValueError(f"forward_greedy: {tok.size} input tokens, expected 1..{self.GREEDY_MAX_IN}")
        if not 1 <= int(n_out) <= self.GREEDY_MAX_OUT:
            raise ValueError(f"forward_greedy: n_out {n_out} not in 1..{self.GREEDY_MAX_OUT}")
        if tok.min() < 0 or tok.max() >= self.config["vocab_size"]:
            raise ValueError(f"forward_greedy: a token is out of range [0, {self.config['vocab_size']})")
        if int(pos) < 0:
            raise ValueError("forward_greedy: negative position")
        if self._h is None:
            raise RuntimeError("Model.forward_greedy: the model is not on a CUDA device (call model.cuda()); this backend has no CPU path")
        out = np.zeros(int(n_out), dtype=np.int32)
        capi.check(capi.lib().xalm_cuda_forward_greedy(self._h, int(tok.size), tok.ctypes.data_as(C.c_void_p), int(pos), int(n_out),
                                                      out.ctypes.data_as(C.c_void_p)))
        return [int(v) for v in out]

    def forward_async(self, token: int, pos: int, mode: int = InferenceMode.OUTPUT_LOGITS) -> None:
        capi.check(capi.lib().xalm_cuda_forward_async(self._h, token, pos, mode))

    def sync(self):
        capi.check(capi.lib().xalm_cuda_sync(self._h))

    # ---- batched decode: one step of several independent sequences (slots of a max_seqs > 1 handle) ---------------------
    @staticmethod
    def _batch_args(seqs, tokens, pos):
        arrs = [np.ascontiguousarray(v, dtype=np.int32).reshape(-1) for v in (seqs, tokens, pos)]
        if not arrs[0].size == arrs[1].size == arrs[2].size:
            raise ValueError("seqs, tokens and pos must have the same length")
        return arrs, [a.ctypes.data_as(C.c_void_p) for a in arrs]

    def forward_batch(self, seqs, tokens, pos, mode: int = InferenceMode.OUTPUT_LOGITS):
        """Slot seqs[i] takes tokens[i] at position pos[i].  OUTPUT_LOGITS -> (n, vocab) logits, row i for seqs[i]; else None."""
        arrs, ptrs = self._batch_args(seqs, tokens, pos)
        n = arrs[0].size
        lg = np.empty((n, self.config["vocab_size"]), dtype=np.float32) if mode == InferenceMode.OUTPUT_LOGITS else None
        capi.check(capi.lib().xalm_cuda_forward_batch(self._h, n, *ptrs, mode, lg.ctypes.data_as(C.c_void_p) if lg is not None else None))
        return lg

    def forward_batch_argmax(self, seqs, tokens, pos) -> list:
        """forward_batch + Sampler.sample_argmax of each row on the device."""
        arrs, ptrs = self._batch_args(seqs, tokens, pos)
        out = np.empty(arrs[0].size, dtype=np.int32)
        capi.check(capi.lib().xalm_cuda_forward_batch_argmax(self._h, arrs[0].size, *ptrs, out.ctypes.data_as(C.c_void_p)))
        return [int(v) for v in out]

    def forward_batch_async(self, seqs, tokens, pos, mode: int = InferenceMode.OUTPUT_LOGITS) -> None:
        arrs, ptrs = self._batch_args(seqs, tokens, pos)
        capi.check(capi.lib().xalm_cuda_forward_batch_async(self._h, arrs[0].size, *ptrs, mode))

    def forward_spans(self, seqs, tokens, pos):
        """forward_batch where a slot may take several consecutive positions in one step (a span, e.g. drafted tokens to
        verify): entry i is slot seqs[i], tokens[i] at pos[i].  Returns the (n, vocab) logits, row i for entry i."""
        arrs, ptrs = self._batch_args(seqs, tokens, pos)
        n = arrs[0].size
        lg = np.empty((n, self.config["vocab_size"]), dtype=np.float32)
        capi.check(capi.lib().xalm_cuda_forward_spans(self._h, n, *ptrs, lg.ctypes.data_as(C.c_void_p)))
        return lg

    def forward_spans_argmax(self, seqs, tokens, pos) -> list:
        """forward_spans + Sampler.sample_argmax of each row on the device."""
        arrs, ptrs = self._batch_args(seqs, tokens, pos)
        out = np.empty(arrs[0].size, dtype=np.int32)
        capi.check(capi.lib().xalm_cuda_forward_spans_argmax(self._h, arrs[0].size, *ptrs, out.ctypes.data_as(C.c_void_p)))
        return [int(v) for v in out]

    @staticmethod
    def _tree_args(tokens, parents):
        arrs = [np.ascontiguousarray(v, dtype=np.int32).reshape(-1) for v in (tokens, parents)]
        if arrs[0].size == 0 or arrs[0].size != arrs[1].size:
            raise ValueError("tokens and parents must have the same, non-zero length")
        return arrs, [a.ctypes.data_as(C.c_void_p) for a in arrs]

    def forward_tree(self, slot: int, tokens, parents, pos: int):
        """One step of a tree of drafted tokens on one slot (tree verification): node i decodes tokens[i] after its ancestors
        (parents[0] == -1, 0 <= parents[i] < i), at position pos + depth(i).  Returns the (n, vocab) logits, row i for node i."""
        arrs, ptrs = self._tree_args(tokens, parents)
        n = arrs[0].size
        lg = np.empty((n, self.config["vocab_size"]), dtype=np.float32)
        capi.check(capi.lib().xalm_cuda_forward_tree(self._h, int(slot), n, *ptrs, int(pos), lg.ctypes.data_as(C.c_void_p)))
        return lg

    def forward_tree_argmax(self, slot: int, tokens, parents, pos: int) -> list:
        """forward_tree + Sampler.sample_argmax of each node's row on the device."""
        arrs, ptrs = self._tree_args(tokens, parents)
        out = np.empty(arrs[0].size, dtype=np.int32)
        capi.check(capi.lib().xalm_cuda_forward_tree_argmax(self._h, int(slot), arrs[0].size, *ptrs, int(pos), out.ctypes.data_as(C.c_void_p)))
        return [int(v) for v in out]

    def tree_accept(self, slot: int, pos: int, nodes) -> None:
        """Move the accepted root-to-node path `nodes` (nodes[0] == 0, increasing) of the tree last verified at pos on this slot
        into rows pos .. pos + len(nodes) - 1.  Enqueue only; nothing when nodes[j] == j for every j."""
        arr = np.ascontiguousarray(nodes, dtype=np.int32).reshape(-1)
        if arr.size == 0:
            raise ValueError("tree_accept: nodes must not be empty")
        capi.check(capi.lib().xalm_cuda_tree_accept(self._h, int(slot), int(pos), arr.size, arr.ctypes.data_as(C.c_void_p)))

    def select_seq(self, seq: int) -> None:
        """The slot forward*, prefill*, read_kv and read_state work on (default 0)."""
        capi.check(capi.lib().xalm_cuda_select_seq(self._h, seq))

    # ---- batched prefill: the per-position loops of main.cpp:94-100 / :244-254 in one pass (tcgen05 GEMMs) ----
    def prefill(self, tokens, pos0: int = 0, want_logits: int = 1, targets=None, fetch_logits: bool = True):
        """Positions pos0..pos0+len(tokens)-1 at once.  want_logits 0: hydrate only -> None; 1: logits of the last
        position (vocab,); 2: all positions (n, vocab).  With `targets` returns (logits, probs) where probs[i] is
        Sampler.sample_prob(targets[i]) at position pos0+i; fetch_logits=False leaves the logits on the device (perplexity
        mode needs only the probabilities).  On a tensor-parallel model this is a collective: every rank calls it with the
        same arguments and gets the full logits and probabilities; a refusal raises the same error on every rank."""
        return self._prefill_call("prefill", tokens, pos0, want_logits, targets, fetch_logits)

    def prefill_window(self, tokens, pos0: int, want_logits: int = 1, targets=None, fetch_logits: bool = True):
        """prefill past the context window, where the KV cache is a ring with two attention sinks: positions
        pos0..pos0+len(tokens)-1 with pos0 >= max_seq_len and len(tokens) <= max_seq_len - 2 (longer runs go in chunks).
        Leaves the KV cache as that many forward() calls would.  Arguments, results and the tensor-parallel collective as for
        prefill()."""
        return self._prefill_call("prefill_window", tokens, pos0, want_logits, targets, fetch_logits)

    def _prefill_call(self, which: str, tokens, pos0: int, want_logits: int, targets, fetch_logits: bool):
        if self._h is None:
            raise RuntimeError(f"Model.{which}: the model is not on a CUDA device (call model.cuda()); this backend has no CPU path")
        tok = np.ascontiguousarray(tokens, dtype=np.int32)
        n = int(tok.size)
        V = self.config["vocab_size"]
        lg = None if want_logits == 0 or not fetch_logits else np.empty(V if want_logits == 1 else (n, V), dtype=np.float32)
        tg = pr = None
        if targets is not None:
            tg = np.ascontiguousarray(targets, dtype=np.int32)
            pr = np.empty(n, dtype=np.float32)
        vp = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        fn = getattr(capi.lib(), "xalm_cuda_" + which)
        capi.check(fn(self._h, vp(tok), n, pos0, want_logits, vp(lg), vp(tg), vp(pr)))
        return (lg, pr) if targets is not None else lg

    def prefill_async(self, tokens: np.ndarray, pos0: int = 0, want_logits: int = 2) -> None:
        capi.check(capi.lib().xalm_cuda_prefill_async(self._h, tokens.ctypes.data_as(C.c_void_p), int(tokens.size), pos0, want_logits))

    def active_bytes(self, pos: int) -> int:
        """Model::active_bytes (model.cpp:12-35) for THIS rank's shard, from the device-side tensor types."""
        b = C.c_longlong(0)
        capi.check(capi.lib().xalm_cuda_active_bytes(self._h, pos, C.byref(b)))
        return b.value

    def last_launch_count(self) -> int:
        n = C.c_int(0)
        capi.check(capi.lib().xalm_cuda_last_launch_count(self._h, C.byref(n)))
        return n.value

    def read_state(self, which: int, n: int) -> np.ndarray:
        out = np.empty(n, dtype=np.float32)
        capi.check(capi.lib().xalm_cuda_read_state(self._h, which, out.ctypes.data_as(C.c_void_p), n))
        return out

    def read_kv(self, layer: int, which: int) -> np.ndarray:
        n = self.config["max_seq_len"] * (self.config["n_kv_heads"] // self.tp_size) * self.config["head_dim"]
        out = np.empty(n, dtype=np.uint16)
        capi.check(capi.lib().xalm_cuda_read_kv(self._h, layer, which, out.ctypes.data_as(C.c_void_p), n))
        return out

    def close(self):
        if self._h is not None:
            capi.lib().xalm_cuda_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def active_bytes_formula(c: dict, bytes_per_weight: float, pos: int, emb_bpw: float | None = None, norm_bytes: int = 4) -> int:
    """SURVEY.md §8d: B(pos) = dim*b_emb + dim*b_norm + vocab*dim*b_cls + L*[2*dim*b_norm + (2*q_dim*dim + 2*kv_dim*dim +
    3*dim*hidden)*b_w + 2*min(max_seq_len,pos+1)*kv_dim*2]."""
    emb_bpw = bytes_per_weight if emb_bpw is None else emb_bpw
    q_dim, kv_dim = c["n_heads"] * c["head_dim"], c["n_kv_heads"] * c["head_dim"]
    b = c["dim"] * emb_bpw + c["dim"] * norm_bytes + c["vocab_size"] * c["dim"] * emb_bpw
    per = 2 * c["dim"] * norm_bytes + (2 * q_dim * c["dim"] + 2 * kv_dim * c["dim"] + 3 * c["dim"] * c["hidden_dim"]) * bytes_per_weight
    per += 2 * min(c["max_seq_len"], pos + 1) * kv_dim * 2
    return int(b + c["n_layers"] * per)


class Sampler:
    """sampler.cpp:3-30 on the host, unchanged — including the FLT_MIN (not lowest) seed of the running max."""

    FLT_MIN = np.float32(np.finfo(np.float32).tiny)

    def __init__(self, config: dict):
        self.vocab_size = config["vocab_size"]

    def sample_argmax(self, state: InferenceState) -> int:
        lg = state.logits()[: self.vocab_size]
        i = int(np.argmax(lg))          # first maximum, like the strict `>` scan
        return i if lg[i] > self.FLT_MIN else 0

    def sample_prob(self, index: int, state: InferenceState) -> float:
        lg = state.logits()[: self.vocab_size]
        mx = max(np.float32(lg.max()), self.FLT_MIN)
        e = np.exp(lg - mx, dtype=np.float32)
        s = np.float32(0)
        s = np.cumsum(e, dtype=np.float32)[-1]      # sequential fp32 sum, as the loop in sampler.cpp:12-14
        return float(np.exp(np.float32(lg[index] - mx), dtype=np.float32) / s)


class Tokenizer:
    """tokenizer.cpp: NUL-separated vocab -> greedy longest-match encode with byte fallback, decode_one."""

    def __init__(self, xalm: X.XalmFile):
        cfg = X.parse_config(xalm.metadata)
        self.bos_id, self.eos_id, self.eot_id = cfg["bos_token_id"], cfg["eos_token_id"], -1
        self.vocab = xalm.tokens()
        self.byte_fallback_start = -1
        for i, t in enumerate(self.vocab):
            if t == b"<0x00>":
                self.byte_fallback_start = i
            elif t in (b"<|eot_id|>", b"<|end|>", b"<|im_end|>"):
                self.eot_id = i
        self._ids = {}
        self._maxlen = 0
        for i, t in enumerate(self.vocab):
            self._ids[t] = i            # later duplicates win, as in the trie build (tokenizer.cpp:56-66)
            self._maxlen = max(self._maxlen, len(t))
        self._prefixes = set()
        for t in self._ids:
            for k in range(1, len(t) + 1):
                self._prefixes.add(t[:k])

    def encode(self, text: str | bytes, encode_bos: bool) -> list:
        data = text.encode("utf-8") if isinstance(text, str) else text
        out = [self.bos_id] if encode_bos else []
        i = 0
        while i < len(data):
            best, l = -1, 0
            while i + l < len(data) and data[i:i + l + 1] in self._prefixes:
                l += 1
                tid = self._ids.get(data[i:i + l], -1)
                if tid >= 0 and len(self.vocab[tid]) == l:
                    best, best_l = tid, l
            if best < 0:
                if self.byte_fallback_start >= 0:
                    out.append(data[i] + self.byte_fallback_start)
                i += 1
            else:
                out.append(best)
                i += best_l
        return out

    def decode_one(self, prev_token: int, token: int) -> bytes:
        piece = self.vocab[token]
        if prev_token == self.bos_id and piece[:1] == b" ":
            return piece[1:]
        if self.byte_fallback_start >= 0 and 0 <= token - self.byte_fallback_start < 256:
            return bytes([token - self.byte_fallback_start])
        return piece
