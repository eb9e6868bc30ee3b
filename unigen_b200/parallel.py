"""Multi-GPU partitioning of the denoiser forward on one 8 x B200 box (NVLink 5 / NVSwitch), one process per GPU.

* Batch data parallelism (BASELINE cfg3): samples are independent -> `dp_shard`; NO data-path collective.
* Ulysses sequence parallelism (cfg4 / long multi-condition sequences): the ONE exchange step of the path is attention.
  Every rank owns S/P rows of the joint [text | image] sequence for all GEMM / LayerNorm / RMSNorm / RoPE work
  (token-local); around attention an all-to-all turns token shards x all heads into all tokens x H/P heads and back
  (4 exchanges per attention: Q, K, V in, O out; 2*S/P*D*2 bytes * (P-1)/P per tensor per rank). QK-RMSNorm and RoPE
  are per token and per head, so they run BEFORE the exchange on the local rows.
  The reference has no sequence parallelism at all (SURVEY.md §5) — this is new design; its contract is numerical
  equality with the single-GPU forward (tests/test_parallel_gpu.py, tests/test_parallel_cpu.py).
  Two implementations of the exchange (`exchange=`):
    "peer" (default) — FUSED into the producing kernels over NVLink peer memory (CUDA IPC pools, `PeerPool`): the QK-RMSNorm +
      RoPE pass stores every head straight into its owner rank's receive buffer (ug_qkv_scatter), the attention epilogue
      stores every output row straight into its owner rank's buffer (ug_attention_bf16_peer), a device-side flag barrier
      separates the phases (2 per attention); all-gathers are peer stores too, so the whole step has no NCCL call, no staging
      copy and replays as ONE CUDA graph per rank.
    "nccl" — staging copy + dist.all_to_all_single x4 per attention (the baseline the fused path is measured against).
  The CoMoE pre-stage (3.6 % of the step, once per step) needs a global top-C token selection per expert; it is computed
  REPLICATED on every rank from an all-gather of the residual stream (28 MB), which keeps routing bit-identical to
  the single-GPU run.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Callable, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from . import _lib, ops
from ._lib import UG_MAX_PEERS, UG_PEER_HANDLE_BYTES, UG_PEER_HEADER_BYTES
from .model import UniGenFlux
from .pvariant import UniCombineFlux


def dp_shard(n_samples: int, world: int, rank: int) -> range:
    """Contiguous block of sample indices owned by `rank` (ragged tails go to the first ranks)."""
    base, rem = divmod(n_samples, world)
    start = rank * base + min(rank, rem)
    return range(start, start + base + (1 if rank < rem else 0))


def sp_row_split(T: int, N: int, world: int, rank: int) -> Tuple[int, int, int, int]:
    """Rows of the joint [text | image] sequence owned by `rank`: (row0, rows, local_text_rows, first_local_image_token)."""
    S = T + N
    if S % world:
        raise ValueError(f"joint sequence {S} is not divisible by the sequence-parallel world size {world}")
    rows = S // world
    row0 = rank * rows
    t_loc = min(max(T - row0, 0), rows)
    return row0, rows, t_loc, max(row0 - T, 0)


class _CudaBuf:
    """`__cuda_array_interface__` carrier so torch can view memory this package allocated (ug_peer_alloc)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = dict(shape=(nbytes,), typestr="|u1", data=(ptr, False), version=2)


def pool_layout(sizes: Sequence[Tuple[str, int]], header: int = UG_PEER_HEADER_BYTES, align: int = 256):
    """Byte offsets of named payload buffers behind the control block: identical on every rank by construction."""
    off, out = header, {}
    for name, nbytes in sizes:
        off = (off + align - 1) // align * align
        out[name] = off
        off += nbytes
    return out, (off + align - 1) // align * align


class PeerPool:
    """A symmetric, peer-mapped device pool: every rank cudaMallocs the same number of bytes, the CUDA IPC handles are
    exchanged once through the process group, and `table` holds this process's mapping of every rank's pool."""

    def __init__(self, group, nbytes: int, device):
        lib = _lib.load()
        self.group, self.world, self.rank = group, dist.get_world_size(group), dist.get_rank(group)
        if self.world > UG_MAX_PEERS:
            raise ops.UgError(f"peer pools support up to {UG_MAX_PEERS} ranks")
        self.nbytes, self.device = int(nbytes), torch.device(device)
        ptr = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(lib.ug_peer_alloc(self.nbytes, C.byref(ptr)), "ug_peer_alloc")
            handle = (C.c_uint8 * UG_PEER_HANDLE_BYTES)()
            _lib.check(lib.ug_peer_export(ptr, handle), "ug_peer_export")
            handles: List[Optional[bytes]] = [None] * self.world
            dist.all_gather_object(handles, bytes(handle), group=group)
            self.table = _lib.PeerTable()
            self.table.world, self.table.rank = self.world, self.rank
            self._opened = []
            for r in range(self.world):
                if r == self.rank:
                    self.table.base[r] = ptr.value
                    continue
                peer = C.c_void_p()
                h = (C.c_uint8 * UG_PEER_HANDLE_BYTES).from_buffer_copy(handles[r])
                _lib.check(lib.ug_peer_open(h, C.byref(peer)), f"ug_peer_open(rank {r})")
                self.table.base[r] = peer.value
                self._opened.append(peer.value)
        self._ptr = ptr.value
        self.local = torch.as_tensor(_CudaBuf(self._ptr, self.nbytes), device=self.device)
        # pinned host mirror of the sticky barrier-error word, refreshed by `poll_error_async` (stream-ordered, no host sync)
        self._err_host = torch.zeros(1, dtype=torch.int32).pin_memory()
        dist.barrier(group=group)  # nobody stores into a pool before every rank has mapped it

    def view(self, offset: int, shape, dtype=torch.bfloat16) -> torch.Tensor:
        n = math.prod(shape) * torch.empty((), dtype=dtype).element_size()
        if offset < UG_PEER_HEADER_BYTES or offset + n > self.nbytes:
            raise ops.UgError("PeerPool.view outside the payload area")
        return self.local[offset:offset + n].view(dtype).view(*shape)

    def barrier(self):
        ops.peer_barrier(self.table)

    def error(self) -> int:
        """Synchronous read of the sticky barrier-error word (0 = every barrier so far completed)."""
        e = C.c_int32()
        _lib.check(_lib.load().ug_peer_error(C.byref(self.table), C.byref(e)), "ug_peer_error")
        return int(e.value)

    def poll_error_async(self):
        """Enqueue a copy of the error word into pinned host memory on the current stream (graph-capturable)."""
        _lib.check(_lib.load().ug_peer_error_async(C.byref(self.table), self._err_host.data_ptr(), ops._stream()), "ug_peer_error_async")

    def raise_on_error(self, sync: bool = False):
        """Raise if a device-side barrier timed out (a rank never arrived: dead peer, or host skew beyond UG_PEER_TIMEOUT_MS).
        sync=False tests the pinned mirror last refreshed by `poll_error_async` — call it after the stream was synchronised
        (e.g. at the start of the next forward); sync=True reads the device word."""
        e = self.error() if sync else int(self._err_host.item())
        if e:
            raise ops.UgError(f"sequence-parallel peer barrier timed out on rank {self.rank} waiting for rank {e - 1}: every result "
                              "since then is invalid (the ranks must be host-synchronised before the first sequence-parallel "
                              "forward; raise UG_PEER_TIMEOUT_MS if ranks legitimately skew by more than the timeout)")

    def __del__(self):  # a dropped pool must not leak its cudaMalloc / IPC mappings (no collective here: peers may be gone)
        try:
            self._release()
        except Exception:  # noqa: BLE001
            pass

    def _release(self):
        lib = _lib.load()
        for p in getattr(self, "_opened", []):
            lib.ug_peer_close(C.c_void_p(p))
        self._opened = []
        if getattr(self, "_ptr", 0):
            self.local = None
            lib.ug_peer_free(C.c_void_p(self._ptr))
            self._ptr = 0

    def close(self):
        lib = _lib.load()
        torch.cuda.synchronize(self.device)
        err = self.error() if self._ptr else 0
        dist.barrier(group=self.group)
        for p in self._opened:
            lib.ug_peer_close(C.c_void_p(p))
        self._opened = []
        if self._ptr:
            self.local = None
            lib.ug_peer_free(C.c_void_p(self._ptr))
            self._ptr = 0
        if err:
            raise ops.UgError(f"peer pool closed with barrier-error word {err} (rank {err - 1} did not arrive at a barrier)")


class UlyssesExchange:
    """The all-to-all pair around attention for ONE sample (B = 1).

    seq_to_heads: local fused QKV rows [S_loc, 3*D] -> (q, k, v) each [S, D/P] (all tokens, this rank's heads)
    heads_to_seq: attention output [S, D/P] -> local rows of the [S_loc, D] (all heads) output view
    `copy` is the strided row-copy primitive (ops.copy on the GPU; a torch fallback is injected by the CPU tests only)."""

    def __init__(self, group, world: int, s_loc: int, d: int, device, dtype, copy: Optional[Callable] = None):
        self.group, self.P, self.s_loc, self.d = group, world, s_loc, d
        self.hd = d // world
        if d % world:
            raise ValueError("hidden size must be divisible by the sequence-parallel world size (whole heads per rank)")
        P, hd = world, self.hd
        self.send = torch.empty(3 * P, s_loc, hd, device=device, dtype=dtype)
        self.recv = torch.empty(3, P * s_loc, hd, device=device, dtype=dtype)
        self.o_full = torch.empty(P * s_loc, hd, device=device, dtype=dtype)
        self.o_recv = torch.empty(P, s_loc, hd, device=device, dtype=dtype)
        self.copy = copy or ops.copy

    def seq_to_heads(self, qkv_local: torch.Tensor):
        """qkv_local: [S_loc, 3*D] view (any row stride). Column block j = which*P + p (which in q,k,v) -> send[j]."""
        P, hd, s_loc = self.P, self.hd, self.s_loc
        src = torch.as_strided(qkv_local, (3 * P, s_loc, hd), (hd, qkv_local.stride(0), 1), qkv_local.storage_offset())
        self.copy(src, self.send)
        for w in range(3):
            dist.all_to_all_single(self.recv[w].view(-1), self.send[w * P:(w + 1) * P].reshape(-1), group=self.group)
        return self.recv[0], self.recv[1], self.recv[2]

    def heads_to_seq(self, out_local: torch.Tensor):
        """o_full [S, hd] (token-major == [P, S_loc, hd]) -> out_local [S_loc, D] view (any row stride)."""
        P, hd, s_loc = self.P, self.hd, self.s_loc
        dist.all_to_all_single(self.o_recv.view(-1), self.o_full.view(-1), group=self.group)
        dst = torch.as_strided(out_local, (P, s_loc, hd), (hd, out_local.stride(0), 1), out_local.storage_offset())
        self.copy(self.o_recv, dst)
        return out_local


class SequenceParallelUniGenFlux(UniGenFlux):
    """UniGenFlux whose main blocks run on S/P rows per rank with Ulysses attention (module docstring). Same public API;
    every rank passes the FULL inputs and receives the FULL velocity (all-gathered)."""

    def __init__(self, arch=None, device="cuda", group=None, exchange: str = "peer", **config):
        super().__init__(arch, device, **config)
        if not dist.is_initialized():
            raise ops.UgError("SequenceParallelUniGenFlux needs an initialised torch.distributed process group")
        if exchange not in ("peer", "nccl"):
            raise ops.UgError("exchange must be 'peer' (fused NVLink peer-memory exchange) or 'nccl' (staged all-to-all)")
        self.sp_group = group
        self.sp_world = dist.get_world_size(group)
        self.sp_rank = dist.get_rank(group)
        if self.arch.num_attention_heads % self.sp_world:
            raise ops.UgError(f"{self.arch.num_attention_heads} heads are not divisible by {self.sp_world} ranks")
        self.exchange = exchange
        # False: this object behaves exactly like the single-GPU UniGenFlux (own workspaces and graphs) — one set of weights
        # serves both the batch-data-parallel and the sequence-parallel measurement of bench.py
        self.sp_enabled = True
        self.sp_prestage = True  # shared-expert blocks of the CoMoE pre-stage sequence-parallel too (peer exchange only)
        self._sp_active = False
        self._xchg = None
        self._pool: Optional[PeerPool] = None
        self._pool_key = None

    def _run_staged(self, key, staged, *args):
        if not self.sp_enabled:
            return super()._run_staged((key, "local"), staged, *args)
        if self.use_consis_module and self.use_shared_expert:
            raise ops.UgError("use_consis_module is not sharded: run with sp_enabled=False (the pre-stage is a small part of the step)")
        if self.linear_dtype != torch.bfloat16:
            raise ops.UgError("fp8-quantised block linears (quantize_fp8) are not sharded: run with sp_enabled=False or a bf16 model")
        if self.exchange != "peer":  # NCCL collectives stay out of graph capture: the staged-exchange baseline runs eagerly
            return self._forward_impl(*args, **staged)
        if self._pool is not None:
            self._pool.raise_on_error()  # barrier-error word mirrored at the end of the previous forward
        return super()._run_staged((key, "sp"), staged, *args)

    def _workspace(self, B: int, N: int, T: int):
        if not self.sp_enabled:
            return super()._workspace(B, N, T)
        # the sequence-parallel workspace re-points AO / CAT / X / HC / MOD into the peer pool: keep it apart from the local one
        return self._cached_workspace((B, N, T, "sp"), lambda: self._make_workspace(B, N, T))

    def check_peer_errors(self):
        """Synchronise and raise if any device-side barrier of the forwards so far timed out (call once per denoise loop)."""
        if self._pool is not None:
            torch.cuda.synchronize(self.device_)
            self._pool.raise_on_error(sync=True)

    def close(self):
        if self._pool is not None:
            self._graphs.clear()
            pool, self._pool, self._pool_key = self._pool, None, None
            pool.close()

    # ---------------------------------------------------------------------------------------------------------
    # exchange = "nccl": staging copy + all_to_all_single around a local attention call
    # ---------------------------------------------------------------------------------------------------------
    def _attend(self, buf, S: int, out: torch.Tensor):
        if not self._sp_active:
            return super()._attend(buf, S, out)
        a = self.arch
        x = self._xchg
        q, k, v = x.seq_to_heads(buf.QKV[0, :S])
        ops.attention(q.unsqueeze(0), k.unsqueeze(0), v.unsqueeze(0), x.o_full.unsqueeze(0), a.num_attention_heads // self.sp_world,
                      a.attention_head_dim, variant=self.attn_variant)
        x.heads_to_seq(out[0])
        return out

    # ---------------------------------------------------------------------------------------------------------
    # exchange = "peer": the exchange is fused into the QK-norm/RoPE pass and the attention epilogue
    # ---------------------------------------------------------------------------------------------------------
    def _peer_setup(self, buf, N: int, T: int, s_loc: int):
        """Pool = [control | RECV [3, S, D/P] | AO [Smax, D] | CAT [S, 5D] | X [S, D] | OUTF [S, in_ch]]; the workspace's AO /
        CAT / X become views of the pool so peers can store attention outputs / gathered rows straight into them."""
        a, D, P = self.arch, self.inner_dim, self.sp_world
        S, Smax = T + N, T + 2 * N
        key = (N, T)
        if self._pool_key != key:
            if self._pool is not None:
                self._graphs.clear()  # captured graphs hold pointers into the old pool
                self._pool.close()
            sizes = [("RECV", 3 * Smax * (D // P) * 2), ("AO", Smax * D * 2), ("CAT", S * 5 * D * 2), ("X", S * D * 2),
                     ("OUTF", S * a.in_channels * 2), ("HC", 2 * N * D * 2), ("MOD", buf.n_mod * D * 4)]
            self._off, total = pool_layout(sizes)
            self._pool = PeerPool(self.sp_group, total, self.device_)
            self._pool_key = key
            self._outf = self._pool.view(self._off["OUTF"], (1, S, a.in_channels))
        pool = self._pool
        buf.AO, buf.CAT, buf.X = (pool.view(self._off["AO"], (1, Smax, D)), pool.view(self._off["CAT"], (1, S, 5 * D)),
                                  pool.view(self._off["X"], (1, S, D)))
        buf.HC = pool.view(self._off["HC"], (1, 2 * N, D))
        buf.MOD = pool.view(self._off["MOD"], (1, buf.n_mod * D), dtype=torch.float32)  # AdaLN table: written by every rank's share
        self._set_sp_rows(S)

    def _set_sp_rows(self, S: int):
        """Contiguous row sharding of an S-row joint sequence: (first global row, rows per rank, S) + the matching view of
        the receive buffer (q, k, v of ALL S tokens for this rank's heads)."""
        if S % self.sp_world:
            raise ops.UgError(f"joint sequence {S} is not divisible by the sequence-parallel world size {self.sp_world}")
        s_loc = S // self.sp_world
        self._sp_rows = (self.sp_rank * s_loc, s_loc, S)
        self._recv = self._pool.view(self._off["RECV"], (3, 1, S, self.inner_dim // self.sp_world))

    def _peer_attention(self, o_name: str, o_row_stride: int):
        """barrier -> attention over this rank's heads of all tokens, output rows stored into their owners' `o_name` buffer ->
        barrier. (barrier 1: every rank's q/k/v stores have landed in RECV; barrier 2: every rank's O stores have landed.)"""
        a, pool = self.arch, self._pool
        _, s_loc, _ = self._sp_rows
        pool.barrier()
        ops.attention_peer(pool.table, self._recv[0], self._recv[1], self._recv[2], a.num_attention_heads // self.sp_world,
                           a.attention_head_dim, self._off[o_name], o_row_stride, s_loc, variant=self.attn_variant)
        pool.barrier()

    def _scatter(self, qkv_rows: torch.Tensor, rms, rope_rows, local_row0: int):
        a = self.arch
        row0, _, S = self._sp_rows
        if self.fuse_qk_norm:  # q / k were normalised and rotated in the projection GEMM's epilogue: the scatter only moves heads
            rms, rope_rows = None, None
        ops.qkv_scatter(self._pool.table, qkv_rows, a.num_attention_heads, a.attention_head_dim, rms, rope_rows, self._off["RECV"], S,
                        row0 + local_row0)

    def _joint_attention(self, buf, B, n_ctx, n_smp, rms_ctx, rms_smp, rope):
        if not (self._sp_active and self.exchange == "peer"):
            return super()._joint_attention(buf, B, n_ctx, n_smp, rms_ctx, rms_smp, rope)
        s = n_ctx + n_smp
        qkv = buf.QKV[0, :s]
        if n_ctx:
            self._scatter(qkv[:n_ctx], rms_ctx, rope[:n_ctx] if rope is not None else None, 0)
        if n_smp:
            self._scatter(qkv[n_ctx:], rms_smp, rope[n_ctx:s] if rope is not None else None, n_ctx)
        self._peer_attention("AO", self.inner_dim)
        return buf.AO[:, :s]

    def _single_attention(self, buf, S: int, rms, rope, out: torch.Tensor):
        if not (self._sp_active and self.exchange == "peer"):
            return super()._single_attention(buf, S, rms, rope, out)
        self._scatter(buf.QKV[0, :S], rms, rope[:S] if rope is not None else None, 0)
        self._peer_attention("CAT", 5 * self.inner_dim)  # `out` is the first D columns of the (peer-mapped) CAT rows
        return out

    def _prestage_sp(self, buf, N, T, x_img, cond_tokens, pooled, cond_pooled, rts_uniform, mods_s0, mods_s1, cond_index,
                     txt_ids, img_ids, cond_ids):
        """CoMoE pre-stage with the two shared-expert blocks SEQUENCE-PARALLEL (they are 95 % of its FLOPs: joint blocks over
        2N and T + 2N tokens); gate / routing / modulated experts stay replicated on the gathered residual stream, so routing is
        bit-identical to the single-GPU run. Row shards of the shared blocks' joint sequences are contiguous:
        shared[0] = [cond | image] (2N rows), shared[1] = [text | image | cond] (T + 2N rows); their outputs are re-gathered
        into the peer-mapped HC buffer by peer stores because the two blocks (and the main blocks) shard differently."""
        a = self.arch
        D, E, C, P, r = self.inner_dim, self.expert_nums, buf.capacity, self.sp_world, self.sp_rank
        gv = self.gemm_variant
        B = 1
        ops.gemm(cond_tokens, self.control_x_embedder_w[0], out=buf.COND, bias=self.control_x_embedder_w[1], variant=gv)
        self._rope(buf.rope0, cond_ids, img_ids)
        self._rope(buf.rope1, txt_ids, img_ids, cond_ids)
        ops.add(x_img, buf.COND, buf.G.view(B, N, D))
        route = ops.moe_route(buf.G, self.gate_wg, rts_uniform, C)
        ops.gemv(cond_pooled, self.exp_mod_w[0], self.exp_mod_b[0], out=buf.MODC.view(B, E * D))
        ops.gemv(pooled, self.exp_mod_w[1], self.exp_mod_b[1], out=buf.MODH.view(B, E * D))
        ops.moe_gather_modulate(buf.COND.view(B * N, D), route["slot_token"], buf.MODC, E, C, N, out=buf.A)
        ops.gemm(buf.A.view(E, C, D), self.exp_w[0], out=buf.YC.view(E, C, D), bias=self.exp_b[0], variant=gv)
        ops.copy(x_img, buf.EH.view(B, N, D))
        ops.moe_gather_modulate(buf.EH, route["slot_token"], buf.MODH, E, C, N, addend=buf.YC, out=buf.A)
        ops.gemm(buf.A.view(E, C, D), self.exp_w[1], out=buf.YH.view(E, C, D), bias=self.exp_b[1], variant=gv)

        def shard(S, n_first):
            """rank's rows of an S-row joint sequence [first stream (n_first rows) | second stream]: (row0, rows, rows of the
            first stream, first local row inside the second stream)."""
            rows = S // P
            row0 = r * rows
            f_loc = min(max(n_first - row0, 0), rows)
            return row0, rows, f_loc, max(row0 - n_first, 0)

        main_rows = self._sp_rows
        loc = self._sp_buf
        if "HL" not in loc:
            loc["HL"] = torch.empty(1, (T + 2 * N) // P + 1, D, device=self.device_, dtype=torch.bfloat16)
        self._sp_active = True
        try:
            # ---- shared[0]: context = condition tokens, sample = image tokens, temb = this condition's temb ----
            S0 = 2 * N
            self._set_sp_rows(S0)
            row0, rows, c_loc, i0 = shard(S0, N)
            s_loc = rows - c_loc
            out_c, out_s = loc["HL"][:, :c_loc], loc["HL"][:, c_loc:rows]
            self._double_block(buf, self.shared[0], mods_s0[0], mods_s0[1], x_img[:, i0:i0 + s_loc], buf.COND[:, row0:row0 + c_loc],
                               out_s, out_c, buf.rope0[row0:row0 + rows])
            # HC = [shared hidden (N) | shared cond (N)] on every rank
            if s_loc:
                ops.peer_bcast_rows(self._pool.table, out_s[0], self._off["HC"], D, i0)
            if c_loc:
                ops.peer_bcast_rows(self._pool.table, out_c[0], self._off["HC"], D, N + row0)
            self._pool.barrier()
            # ---- shared[1]: context = control text, sample = [hidden | cond], temb = control_temb, context output discarded ----
            S1 = T + 2 * N
            self._set_sp_rows(S1)
            row0, rows, t_loc, h0 = shard(S1, T)
            h_loc = rows - t_loc
            hl = loc["HL"][:, :h_loc]
            self._double_block(buf, self.shared[1], mods_s1[0], mods_s1[1], buf.HC[:, h0:h0 + h_loc], buf.CENC[:, row0:row0 + t_loc],
                               hl, None, buf.rope1[row0:row0 + rows])
            self._pool.barrier()  # every rank has finished READING its HC rows before anyone overwrites them
            if h_loc:
                ops.peer_bcast_rows(self._pool.table, hl[0], self._off["HC"], D, h0)
            self._pool.barrier()
        finally:
            self._sp_active = False
            self._sp_rows = main_rows
            self._set_sp_rows(main_rows[2])
        hc_h, hc_c = buf.HC[:, :N], buf.HC[:, N:]
        ops.moe_combine(buf.YH, route, C, buf.EH)
        ops.moe_combine(buf.YC, route, C, buf.EC)
        if cond_index == 0:
            ops.add(hc_h, buf.EH.view(B, N, D), buf.CIN)
        else:
            ops.add(buf.CIN, hc_h, buf.CIN)
            ops.add(buf.CIN, buf.EH.view(B, N, D), buf.CIN)
        ops.add(buf.CIN, hc_c, buf.CIN)
        ops.add(buf.CIN, buf.EC.view(B, N, D), buf.CIN)
        return route

    def _gather_rows(self, local: torch.Tensor, name: str, full: torch.Tensor):
        """all-gather of [s_loc, d] row shards into the [S, d] buffer `name` of every rank."""
        if self.exchange == "peer":
            ops.peer_bcast_rows(self._pool.table, local[0], self._off[name], full.shape[-1], self._sp_rows[0])
            self._pool.barrier()
        else:
            dist.all_gather_into_tensor(full.view(-1), local.reshape(-1), group=self.sp_group)

    def _forward_impl(self, conditioning_scale, hs, es, pooled, timestep, guidance, txt_ids, img_ids, **cond):
        if not self.sp_enabled:
            return UniGenFlux._forward_impl(self, conditioning_scale, hs, es, pooled, timestep, guidance, txt_ids, img_ids, **cond)
        a = self.arch
        P, rank = self.sp_world, self.sp_rank
        n_cond = self.condition_nums
        cs = [ops.to_bf16(cond[f"cs{c}"].contiguous()) for c in range(n_cond)]
        cond_pooled = [cond[f"cp{c}"] for c in range(n_cond)]
        condition_ids = [cond[f"cid{c}"] for c in range(n_cond)]
        rts_uniform = [cond[f"u{c}"] for c in range(n_cond)]
        D = self.inner_dim
        B, N, _ = hs.shape
        T = es.shape[1]
        S = T + N
        if B != 1:
            raise ops.UgError("sequence parallelism shards ONE sample across ranks (use batch data-parallelism for B > 1)")
        row0, s_loc, t_loc, i0 = sp_row_split(T, N, P, rank)
        n_img = s_loc - t_loc
        buf = self._workspace(B, N, T)
        dev = self.device_
        n0 = ops.launch_count()
        if getattr(self, "_sp_key", None) != (N, T):
            if self.exchange == "nccl":
                self._xchg = UlyssesExchange(self.sp_group, P, s_loc, D, dev, torch.bfloat16)
            self._sp_buf = dict(XL=torch.empty(1, s_loc, D, device=dev, dtype=torch.bfloat16),
                                NOL=torch.empty(1, s_loc, D, device=dev, dtype=torch.bfloat16),
                                OUTL=torch.empty(1, s_loc, a.in_channels, device=dev, dtype=torch.bfloat16))
            if self.exchange == "nccl":
                self._sp_buf["OUTF"] = torch.empty(1, S, a.in_channels, device=dev, dtype=torch.bfloat16)
            self._sp_key = (N, T)
        if self.exchange == "peer":
            self._peer_setup(buf, N, T, s_loc)
            self._sp_buf["OUTF"] = self._outf
        XL = self._sp_buf["XL"]
        xl_txt, xl_img = XL[:, :t_loc], XL[:, t_loc:]
        hs, es = ops.to_bf16(hs.contiguous()), ops.to_bf16(es.contiguous())
        gv = self.gemm_variant

        # ---- embeddings on the local rows only ----
        if n_img:
            ops.gemm(hs[:, i0:i0 + n_img], self.x_embedder_w[0], out=xl_img, bias=self.x_embedder_w[1], variant=gv)
        if t_loc:
            ops.gemm(es[:, row0:row0 + t_loc], self.context_embedder_w[0], out=xl_txt, bias=self.context_embedder_w[1], variant=gv)
        self._conditioning_vectors(buf, B, timestep, guidance, pooled, cond_pooled)
        self._rope(buf.rope, txt_ids, img_ids)
        rope_loc = buf.rope[row0:row0 + s_loc]

        # ---- AdaLN vectors of every block (step constants). exchange="peer": the ~10 GB weight stream is SHARDED — every rank
        # runs 1/P of the grouped-GEMV work list and stores its results into every rank's peer-mapped MOD table (the all-gather
        # is the stores themselves), one barrier; exchange="nccl" (baseline): replicated, as on one GPU ----
        main_stream = torch.cuda.current_stream()
        if self.exchange == "peer":
            mp = self._mod_plans(buf, pool=self._pool)
            ops.gemv_grouped(mp.all, rank, P)
            self._pool.barrier()
            side, mods_joined = None, True
        else:
            mp = self._mod_plans(buf)
            ops.gemv_grouped(mp.early)
            side = self._side_stream if self.overlap_mod_gemv else None
            if side is not None:
                side.wait_stream(main_stream)
            with torch.cuda.stream(side if side is not None else main_stream):
                ops.gemv_grouped(mp.late)
            mods_joined = side is None
        m_double, m_cdouble, m_single, m_csingle = mp.m_double, mp.m_cdouble, mp.m_single, mp.m_csingle
        mods_s0, mods_s1, m_out = mp.mods_s0, mp.mods_s1, mp.m_out
        nd = len(self.double)

        # ---- double blocks on token shards ----
        route = None
        n_cd = len(self.ctrl_double)
        cenc_loc = None
        self._sp_active = True
        try:
            for i, w in enumerate(self.double):
                if i == 1 and not mods_joined:
                    main_stream.wait_stream(side)
                    mods_joined = True
                self._double_block(buf, w, m_double[i][0], m_double[i][1], xl_img, xl_txt, xl_img, xl_txt, rope_loc)
                j = int(i / (len(self.double) / n_cd))
                if route is None:
                    # CoMoE pre-stage, replicated: gather the residual stream once, route / run experts on every rank
                    self._sp_active = False
                    self._gather_rows(XL, "X", buf.X)
                    x_txt, x_img = buf.X[:, :T], buf.X[:, T:]
                    ops.gemm(x_txt, self.control_context_embedder_w[0], out=buf.CENC, bias=self.control_context_embedder_w[1], variant=gv)
                    for c in range(n_cond):
                        if self.exchange == "peer" and self.sp_prestage and (2 * N) % P == 0 and (T + 2 * N) % P == 0:
                            route = self._prestage_sp(buf, N, T, x_img, cs[c], pooled, cond_pooled[c], rts_uniform[c], mods_s0[c],
                                                      mods_s1, c, txt_ids, img_ids, condition_ids[c])
                        else:
                            route = self._prestage(buf, B, N, T, x_img, cs[c], pooled, cond_pooled[c], rts_uniform[c], mods_s0[c],
                                                   mods_s1, c, txt_ids, img_ids, condition_ids[c])
                    self._sp_active = True
                    ctrl_in = buf.CIN[:, i0:i0 + n_img]
                    cenc_loc = buf.CENC[:, row0:row0 + t_loc]
                else:
                    ctrl_in = xl_img
                ch = buf.CH[:, :n_img]
                self._double_block(buf, self.ctrl_double[j], m_cdouble[j][0], m_cdouble[j][1], ctrl_in, cenc_loc, ch, None, rope_loc)
                if n_img:
                    wa = self.add_double[j]
                    ops.gemm(ch, wa[0], out=xl_img, bias=wa[1], alpha=float(conditioning_scale), residual=xl_img, variant=gv)
            if not mods_joined:
                main_stream.wait_stream(side)
                mods_joined = True
            # ---- single blocks ----
            n_cs = len(self.ctrl_single)
            csl = buf.CS[:, :s_loc]
            for i, w in enumerate(self.single):
                self._single_block(buf, w, m_single[i], XL, XL, rope_loc)
                if n_cs:
                    j = int(i / (len(self.single) / n_cs))
                    self._single_block(buf, self.ctrl_single[j], m_csingle[j], XL, csl, rope_loc)
                    wa = self.add_single[j]
                    if self.single_block_control_method == "overall_add":
                        ops.gemm(csl, wa[0], out=XL, bias=wa[1], alpha=float(conditioning_scale), residual=XL, variant=gv)
                    elif n_img:
                        ops.gemm(csl[:, t_loc:], wa[0], out=xl_img, bias=wa[1], alpha=float(conditioning_scale), residual=xl_img, variant=gv)
        finally:
            self._sp_active = False
        # ---- norm_out + proj_out on the local rows, then gather the velocity ----
        sb = self._sp_buf
        ops.ln_modulate(XL, sb["NOL"], m_out[1], m_out[0])
        ops.gemm(sb["NOL"], self.proj_out_w[0], out=sb["OUTL"], bias=self.proj_out_w[1], variant=gv)
        self._gather_rows(sb["OUTL"], "OUTF", sb["OUTF"])
        if self.exchange == "peer":
            self._pool.poll_error_async()
        self._last_route = route
        ops.note_capture_launches(ops.launch_count() - n0)
        return sb["OUTF"][:, T:], dict(moe_loss=route["l_aux"][0] * 0.1), dict(expert_counts=route["exp_counts"])


class SequenceParallelUniCombineFlux(UniCombineFlux):
    """P-variant (LoRA-switched joint blocks, all condition tokens in every block — BASELINE cfg4's "~17 k tokens") with
    SEGMENT-SHARDED Ulysses attention: every rank holds 1/P of the text, image and each condition stream, so the local
    sequence keeps the [txt | img | c_1 .. c_n] segment structure (all per-segment switches — LoRA group, AdaLN vectors,
    gates — work unchanged on local bounds = global bounds / P). Around attention the exchange is fused into the kernels over
    NVLink peer memory exactly as in `SequenceParallelUniGenFlux` (exchange="peer"): per segment, ug_qkv_scatter normalises /
    rotates q,k and stores heads into their owner rank's receive buffer at the segment's GLOBAL rows; ug_attention_bf16_peer
    runs the segment-visibility mask on global bounds and stores each output row into its owner's AO / CAT rows.
    Every rank passes the FULL inputs and receives the FULL velocity. Numerical contract: bit-identical to the single-GPU
    `UniCombineFlux.forward` (tools/sp_check_pvariant.py)."""

    def __init__(self, arch=None, device="cuda", group=None, **kw):
        super().__init__(arch, device, **kw)
        if not dist.is_initialized():
            raise ops.UgError("SequenceParallelUniCombineFlux needs an initialised torch.distributed process group")
        self.sp_group, self.sp_world, self.sp_rank = group, dist.get_world_size(group), dist.get_rank(group)
        if self.arch.num_attention_heads % self.sp_world:
            raise ops.UgError(f"{self.arch.num_attention_heads} heads are not divisible by {self.sp_world} ranks")
        self._pool: Optional[PeerPool] = None
        self._pool_key = None
        self.use_cuda_graph = False
        self._graphs = {}
        self.sp_enabled = True  # False: behaves exactly like the single-GPU UniCombineFlux (same weights; bench.py's 1-GPU leg)

    def _workspace(self, B, S_loc):
        buf = super()._workspace(B, S_loc)
        if not self.sp_enabled:
            return buf
        if B != 1:
            raise ops.UgError("sequence parallelism shards ONE sample across ranks (use batch data-parallelism for B > 1)")
        a, D, P = self.arch, self.inner_dim, self.sp_world
        S = S_loc * P
        if self._pool_key != S_loc:
            if self._pool is not None:
                self._graphs.clear()  # captured graphs hold pointers into the old pool
                self._pool.close()
            n_max = S  # velocity rows <= S
            sizes = [("RECV", 3 * S * (D // P) * 2), ("AO", S_loc * D * 2), ("CAT", S_loc * 5 * D * 2), ("OUTF", n_max * a.in_channels * 2),
                     ("PMOD", self._mod_layout(B, self.groups - 1)[-1] * 4)]  # AdaLN tables: every rank computes 1/P, stores to all
            self._off, total = pool_layout(sizes)
            self._pool = PeerPool(self.sp_group, total, self.device_)
            self._pool_key = S_loc
            self._recv = self._pool.view(self._off["RECV"], (3, 1, S, D // P))
        buf.AO, buf.CAT = self._pool.view(self._off["AO"], (1, S_loc, D)), self._pool.view(self._off["CAT"], (1, S_loc, 5 * D))
        return buf

    def _mods(self, buf, B: int, n: int):
        """AdaLN tables SHARDED over the ranks: each rank runs 1/P of every grouped-GEMV launch and stores its results into every
        rank's peer-mapped table (the all-gather is the stores themselves); a barrier before the accumulating LoRA launch (it
        reads the down-projections and the running table values other ranks produced) and one after it."""
        if not self.sp_enabled:
            return super()._mods(buf, B, n)
        P, r, pool = self.sp_world, self.sp_rank, self._pool
        total = self._mod_layout(B, n)[-1]
        flat = pool.view(self._off["PMOD"], (total,), dtype=torch.float32)
        mp = self._mod_plans(buf, B, n, flat=flat, pool=pool)
        mp.tembs[0].copy_(buf.temb)
        for j in range(n):
            mp.tembs[1 + j].copy_(buf.ctemb)
        ops.silu(mp.tembs, mp.stembs)
        ops.gemv_grouped(mp.main, r, P)
        ops.gemv_grouped(mp.ctx, r, P)
        pool.barrier()
        ops.gemv_grouped(mp.lora, r, P)
        pool.barrier()
        return mp

    def _attention(self, buf, parts, out_name: str, bounds, vis):
        if not self.sp_enabled:
            return super()._attention(buf, parts, out_name, bounds, vis)
        a, D, P, pool = self.arch, self.inner_dim, self.sp_world, self._pool
        H, dh = a.num_attention_heads, a.attention_head_dim
        gbounds = [b * P for b in bounds]
        S = gbounds[-1]
        qkv = buf.QKV[0]
        for s in range(len(bounds) - 1):  # one scatter per local segment shard -> its global rows
            lo, hi = bounds[s], bounds[s + 1]
            if hi == lo:
                continue
            rms = next(w for plo, phi, w in parts if plo <= lo and hi <= phi)
            fused = self._fused_qk()  # q / k already normalised and rotated by the projection GEMM: the scatter only moves heads
            ops.qkv_scatter(pool.table, qkv[lo:hi], H, dh, None if fused else rms, None if fused else buf.rope[lo:hi],
                            self._off["RECV"], S, gbounds[s] + self.sp_rank * (hi - lo))
        pool.barrier()
        ops.attention_peer(pool.table, self._recv[0], self._recv[1], self._recv[2], H // P, dh, self._off[out_name],
                           D if out_name == "AO" else 5 * D, 0, seg_bounds=gbounds, seg_visible=vis, variant=self.attn_variant)
        pool.barrier()

    def _forward_local(self, hs, cl, cids, es, pooled, timestep, img_ids, txt_ids, condition_types, c_t, N):
        out_loc = super().forward(hs, cl, cids, condition_types, es, pooled, timestep, img_ids, txt_ids, c_t=c_t)
        n_loc = out_loc.shape[1]
        ops.peer_bcast_rows(self._pool.table, out_loc[0], self._off["OUTF"], self.arch.in_channels, self.sp_rank * n_loc)
        self._pool.barrier()
        self._pool.poll_error_async()
        return self._pool.view(self._off["OUTF"], (1, N, self.arch.in_channels))

    def check_peer_errors(self):
        """Synchronise and raise if any device-side barrier of the forwards so far timed out (call once per denoise loop)."""
        if self._pool is not None:
            torch.cuda.synchronize(self.device_)
            self._pool.raise_on_error(sync=True)

    def close(self):
        if self._pool is not None:
            self._graphs.clear()
            pool, self._pool, self._pool_key = self._pool, None, None
            pool.close()

    @torch.no_grad()
    def forward(self, hidden_states, condition_latents, condition_ids, condition_types, encoder_hidden_states,
                pooled_projections, timestep, img_ids, txt_ids, c_t: float = 0.0, **kwargs):
        if not self.sp_enabled:
            return UniCombineFlux.forward(self, hidden_states, condition_latents, condition_ids, condition_types,
                                          encoder_hidden_states, pooled_projections, timestep, img_ids, txt_ids, c_t=c_t, **kwargs)
        if self.linear_dtype != torch.bfloat16:
            raise ops.UgError("fp8-quantised block linears (quantize_fp8) are not sharded: run with sp_enabled=False or a bf16 model")
        P, r = self.sp_world, self.sp_rank
        dev = self.device_
        if self._pool is not None:
            self._pool.raise_on_error()  # barrier-error word mirrored at the end of the previous forward
        self._sync_lora()  # outside any graph capture / replay: hook changes rewrite the operand stacks in place

        def shard(t, dim):
            n = t.shape[dim]
            if n % P:
                raise ops.UgError(f"segment of {n} tokens is not divisible by the sequence-parallel world size {P}")
            return t.narrow(dim, r * (n // P), n // P).to(dev).contiguous()

        N = hidden_states.shape[1]
        local = dict(hs=shard(hidden_states, 1), es=shard(encoder_hidden_states, 1), pooled=pooled_projections.to(dev),
                     timestep=timestep.to(dev), img_ids=shard(img_ids, 0), txt_ids=shard(txt_ids, 0))
        for j, (c, ci) in enumerate(zip(condition_latents, condition_ids)):
            local[f"cl{j}"], local[f"cid{j}"] = shard(c, 1), shard(ci, 0)
        n = len(condition_latents)

        def run(t):
            return self._forward_local(t["hs"], [t[f"cl{j}"] for j in range(n)], [t[f"cid{j}"] for j in range(n)], t["es"], t["pooled"],
                                       t["timestep"], t["img_ids"], t["txt_ids"], list(condition_types), c_t, N)

        if not self.use_cuda_graph or self.trace is not None:
            return self._own(run(local))
        key = (tuple((k, tuple(v.shape), v.dtype) for k, v in local.items()), tuple(condition_types), float(c_t))
        g = self._graphs.get(key)
        if g is None:
            static = {k: v.clone() for k, v in local.items()}
            run(static)  # warm-up: pool creation (IPC handle exchange), workspace allocation
            torch.cuda.synchronize()
            n0 = ops.launch_count()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = run(static)
            g = self._graphs[key] = (graph, static, out, ops.launch_count() - n0)
        graph, static, out, n_launch = g
        for k, v in local.items():
            static[k].copy_(v)
        graph.replay()
        ops.add_launches(n_launch)
        return self._own(out)

    @staticmethod
    def _own(out: torch.Tensor) -> torch.Tensor:
        """The velocity is gathered into the peer pool (freed / rewritten by later forwards): return a copy the caller owns."""
        return ops.copy(out, torch.empty(out.shape, device=out.device, dtype=out.dtype))
