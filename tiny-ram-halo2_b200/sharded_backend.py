"""plonk.create_proof on several GPUs of one box (SURVEY.md 8(e); BASELINE.json configs[4]): one process per GPU, every process
runs the SAME host logic on the same witness with the same RNG stream (ShardedRng: rank 0's OS seed, broadcast), so the
transcript is replicated and no rank waits for another's challenges.  The COMPUTE of every heavy phase is divided, the RESULTS
are replicated, so that the host logic above never has to know where a polynomial lives:

  * commitments (best_multiexp): the columns of every commit_lagrange_many / commit_many batch go round-robin over the ranks
    (parallel.shard_columns), the 64-byte affine results are all_gathered;
  * lagrange_to_coeff: a batch's columns are owned in contiguous blocks, each rank transforms its block inside the proof's
    polynomial arena and ONE in-place all_gather fills the other blocks (k = 20: 15.5 GiB per proof over NVLink);
  * lookups: lookup i (compress, permute_expression_pair, later its grand product) belongs to rank i // ceil(L / G); the permuted
    columns and the Z columns are all_gathered in place;
  * the permutation argument: every chunk's grand product is computed from 1 by its owner, the chunk-end values are
    all_gathered (a few scalars) and each chunk is scaled by the product of its predecessors' ends -- exactly the chain
    z_i[0] = z_{i-1}[u] halo2 builds sequentially -- then the Z columns are all_gathered;
  * the quotient: every rank expands ITS block of coefficient columns on a coset (one size-n NTT per column), an all-to-all
    hands rank r the rows [r n / G - halo, (r + 1) n / G + halo) of every column, rank r runs the quotient program on its n / G
    rows (trp_dev_quotient_eval_rows) -- so j - 1 = 5 cosets load 2, 4 or 8 devices evenly, NTTs and program alike -- and the
    n-value results are all_gathered; every rank recovers h(X).  Key-material cosets are cached per rank as row slices.

Replicated: openings' evaluations, multiopen's linear combinations, Kate divisions and the IPA (every rank holds every
coefficient polynomial after the all_gathers).  The proof bytes are identical on every rank and identical to the one-GPU proof.

ShardedCommits is a mixin over any backend of plonk.create_proof, so the commit partition is tested on CPU over gloo with the
oracle's PythonBackend (tests/test_parallel_cpu.py); the exchange helpers (parallel.py) are gloo-tested on CPU tensors."""
from __future__ import annotations

import os

import numpy as np

from . import parallel
from . import poly as P
from .plonk import GpuBackend


class ShardedCommits:
    """mixin: commit_lagrange_many / commit_many sharded by column.  Needs self.dist (torch.distributed or None) and
    self.comm_device ("cuda" for nccl, "cpu" for gloo)."""
    dist = None
    comm_device = "cpu"

    def _sharded_points(self, commit_many, vecs, blinds):
        d = self.dist
        if d is None or d.get_world_size() == 1 or not len(vecs):
            return commit_many(vecs, blinds)
        import torch
        world, rank = d.get_world_size(), d.get_rank()
        mine = parallel.shard_columns(len(vecs), world, rank)
        local = commit_many([vecs[i] for i in mine], [blinds[i] for i in mine]) if mine else []
        per_rank = (len(vecs) + world - 1) // world
        buf = np.zeros((per_rank, 65), dtype=np.uint8)               # flag, x, y (32-byte little-endian); flag 0 = identity
        for j, pt in enumerate(local):
            if pt is not None:
                buf[j, 0] = 1
                buf[j, 1:33] = np.frombuffer(pt[0].to_bytes(32, "little"), dtype=np.uint8)
                buf[j, 33:65] = np.frombuffer(pt[1].to_bytes(32, "little"), dtype=np.uint8)
        t = torch.from_numpy(buf).to(self.comm_device)
        parts = [torch.empty_like(t) for _ in range(world)]
        d.all_gather(parts, t)
        parts = [p.cpu().numpy() for p in parts]
        out = []
        for c in range(len(vecs)):
            r, j = parallel.owner_of_column(c, world)
            row = parts[r][j]
            out.append((int.from_bytes(row[1:33].tobytes(), "little"), int.from_bytes(row[33:65].tobytes(), "little")) if row[0] else None)
        return out

    def commit_lagrange_many(self, vecs, blinds, **kw):
        return self._sharded_points(lambda v, b: super(ShardedCommits, self).commit_lagrange_many(v, b, **kw), vecs, blinds)

    def commit_many(self, vecs, blinds):
        return self._sharded_points(super().commit_many, vecs, blinds)


class ShardedRng:
    """The caller's RNG of a multi-GPU create_proof: every rank must draw the SAME stream.  Rank 0 takes 32 bytes from the OS,
    the seed is broadcast, and the stream is AES-256-CTR keyed by it (a CSPRNG; `cryptography` is in the image).
    rand() reads 64 bytes of the scalar stream (counter block 0 onwards) and reduces them mod p -- pasta's Field::random =
    from_u512 of eight next_u64.  vector(n), the bulk draw of a random polynomial, is draw number i of its own stream (nonce
    i + 1): n x 32 bytes with the top two bits cleared, used as Montgomery limbs (uniform below 2^254, 2^-128 from uniform mod p).
    Bulk draws do not depend on how many scalars were drawn before them, so prefetch(n, count) can produce the next `count` of
    them on a worker thread while the GPU is busy (32 MiB of keystream per polynomial at k = 20)."""

    def __init__(self, p: int, dist=None, device="cpu", seed: bytes = None):
        import os
        import torch
        if seed is None:
            seed = os.urandom(32)
        if dist is not None and dist.get_world_size() > 1:
            t = torch.tensor(list(seed), dtype=torch.uint8, device=device)
            dist.broadcast(t, src=0)
            seed = bytes(t.cpu().tolist())
        self.seed, self.p = seed, p
        self._enc = self._stream(0)
        self._buf, self._off = b"", 0
        self.draws = 0
        self._vec_index = 0
        self._pending = {}
        self._pool = None

    def _stream(self, nonce: int):
        from cryptography.hazmat.primitives.ciphers import Cipher, algorithms, modes
        return Cipher(algorithms.AES(self.seed), modes.CTR(nonce.to_bytes(8, "big") + b"\0" * 8)).encryptor()

    def __call__(self):
        self.draws += 1
        if self._off + 64 > len(self._buf):                  # keystream in 64 KiB blocks (a proof draws ~2 800 scalars)
            self._buf, self._off = self._enc.update(bytes(1 << 16)), 0
        v = int.from_bytes(self._buf[self._off:self._off + 64], "little") % self.p
        self._off += 64
        return v

    def bulk_key(self) -> bytes:
        """32 bytes of the scalar stream: the key a device-resident backend expands into a random polynomial
        (plonk.GpuBackend.random_vec -> trp_dev_random_field), instead of 64 n bytes of keystream crossing PCIe"""
        if self._off + 32 > len(self._buf):
            self._buf, self._off = self._enc.update(bytes(1 << 16)), 0
        k = self._buf[self._off:self._off + 32]
        self._off += 32
        self.draws += 1
        return k

    def _make_vector(self, index: int, n: int):
        a = np.frombuffer(self._stream(index + 1).update(bytes(32 * n)), dtype=np.uint64).reshape(n, 4).copy()
        a[:, 3] &= np.uint64((1 << 62) - 1)
        return a

    def prefetch(self, n: int, count: int):
        from concurrent.futures import ThreadPoolExecutor
        if self._pool is None:
            self._pool = ThreadPoolExecutor(max_workers=1)
        for i in range(self._vec_index, self._vec_index + count):
            if (i, n) not in self._pending:
                self._pending[(i, n)] = self._pool.submit(self._make_vector, i, n)

    def vector(self, n):
        i = self._vec_index
        self._vec_index += 1
        self.draws += n
        fut = self._pending.pop((i, n), None)
        return fut.result() if fut is not None else self._make_vector(i, n)


class ShardedGpuBackend(ShardedCommits, GpuBackend):
    """plonk.GpuBackend on this process's GPU + the partitions above over `dist` (an initialised NCCL process group)"""
    comm_device = "cuda"
    HALO = 16                              # rows kept either side of a row slice (rotations of +-16 rows: TinyRAM needs -6 .. +1)

    def __init__(self, ctx, k, cs_degree, dist=None, params=None):
        self.dist = dist if (dist is not None and dist.get_world_size() > 1) else None
        self.world = self.dist.get_world_size() if self.dist else 1
        self.rank = self.dist.get_rank() if self.dist else 0
        super().__init__(ctx, k, cs_degree, params=params)
        if self.world > 1 and self.n % self.world:
            raise ValueError("the number of GPUs must divide 2^k")
        self._xbuf = {}                    # persistent exchange buffers
        self._pending = []                 # all_gathers of coefficient polynomials still in flight (lagrange_to_coeff_many)

    # -- small helpers ------------------------------------------------------------------------------------------------------------
    def _buf(self, name, shape):
        t = self.torch
        cur = self._xbuf.get(name)
        if cur is None or tuple(cur.shape) != tuple(shape):
            self._xbuf[name] = None
            cur = self._xbuf[name] = t.empty(shape, dtype=t.int64, device="cuda")
        return cur

    def _arena_padding(self):
        return self.world                  # the in-place all_gather of a batch writes whole blocks

    def close(self):
        self._drain()
        self._xbuf.clear()
        super().close()

    def _drain(self):
        """wait for the exchanges lagrange_to_coeff_many left in flight: from here on every rank holds every coefficient polynomial"""
        for w in self._pending:
            w.wait()
        self._pending = []

    # everything that reads coefficient polynomials other ranks produced waits for their arrival first
    def begin_proof(self, n_polys):
        self._drain()
        return super().begin_proof(n_polys)

    def eval_polynomial(self, v, x):
        self._drain()
        return super().eval_polynomial(v, x)

    def linear_combination(self, vs, scalars):
        """multiopen's q polynomials (sum_j x_1^j p_j over up to ~700 polynomials): every rank combines a block of the terms, the
        partial sums are all_gathered (world x 32 MiB at k = 20) and added -- field addition is exact, so the result is the same
        canonical vector whatever the grouping"""
        self._drain()
        if self.world == 1 or len(vs) < 4 * self.world:
            return super().linear_combination(vs, scalars)
        per, lo, hi = parallel.block_range(len(vs), self.world, self.rank)
        part = super().linear_combination(vs[lo:hi], scalars[lo:hi]) if hi > lo else self._new(zero=True)
        parts = self._buf("lincomb_parts", (self.world, self.n, 4))
        self.dist.all_gather_into_tensor(parts, part)
        return super().linear_combination([parts[r] for r in range(self.world)], [1] * self.world)

    def kate_division(self, v, b):
        self._drain()
        return super().kate_division(v, b)

    def commit_many(self, vecs, blinds):
        self._drain()
        return super().commit_many(vecs, blinds)

    def ipa_create_proof(self, rand, transcript, p_poly, p_blind, x_3):
        self._drain()
        return super().ipa_create_proof(rand, transcript, p_poly, p_blind, x_3)

    def _ipa_dist(self):
        w = self.world
        return self.dist if (w > 1 and w & (w - 1) == 0 and w <= self.n and os.environ.get("TRP_IPA_SHARDED", "1") != "0") else None

    # -- lagrange_to_coeff: blocks of columns, one in-place all_gather --------------------------------------------------------------
    def lagrange_to_coeff_many(self, vs):
        k = len(vs)
        if self.world == 1 or not self._arena_on or k < self.world:
            return super().lagrange_to_coeff_many(vs)
        first = self._arena_used
        if first + k > self._arena.shape[0]:
            return super().lagrange_to_coeff_many(vs)
        # rank r transforms columns [r * per, (r + 1) * per) of the batch; the k mod world columns left over are transformed by
        # EVERY rank (at most world - 1 redundant transforms), so the exchange covers whole blocks only and never writes outside the
        # batch's own slots -- it stays in flight while the next batch fills the slots right behind it
        per, main, lo, hi = parallel.whole_block_range(k, self.world, self.rank)
        out = []
        for i, v in enumerate(vs):
            c = self._arena[first + i]
            self._arena_slot[id(c)] = (first + i, c)
            if lo <= i < hi or i >= main:
                c.copy_(v)
            out.append(c)
        self._arena_used += k
        self.ctx.check(self.lib.trp_dev_lagrange_to_coeff(self.dom.handle, self._arena[first + lo].data_ptr(), hi - lo))
        if k > main:
            self.ctx.check(self.lib.trp_dev_lagrange_to_coeff(self.dom.handle, self._arena[first + main].data_ptr(), k - main))
        # the other ranks' blocks are not read before the quotient (which waits: _drain), so the exchange runs on NCCL's stream
        # underneath the next phases' kernels -- 15.5 GiB per proof at k = 20, a tenth of the step on 8 GPUs if it is waited for here
        w = parallel.all_gather_blocks_inplace(self._arena[first:first + main], per, self.dist, async_op=True)
        if w is not None:
            self._pending.append(w)
        return out

    # -- openings: every rank evaluates a block of the polynomials, the values are all_gathered --------------------------------------------
    def eval_polynomials_at(self, vs, x):
        self._drain()
        if self.world == 1 or len(vs) < 4 * self.world:
            return super().eval_polynomials_at(vs, x)
        per, lo, hi = parallel.block_range(len(vs), self.world, self.rank)
        vals = self.torch.zeros((per * self.world, 4), dtype=self.torch.int64, device="cuda")
        if hi > lo:
            tab = (self.ct.c_void_p * (hi - lo))(*[v.data_ptr() for v in vs[lo:hi]])
            self.ctx.check(self.lib.trp_dev_eval_polynomials_at(self.ctx.handle, 0, tab, self.n, hi - lo, self._m(x), vals[lo].data_ptr()))
        parallel.all_gather_blocks_inplace(vals, per, self.dist)
        return self._ints(vals[:len(vs)].cpu().numpy().view(self.np.uint64))

    # -- lookups: owned in blocks -------------------------------------------------------------------------------------------------------
    def lookups_commit_permuted(self, lookups, theta, values_of, usable, bf, rand):
        L = len(lookups)
        draws = []
        for _ in range(L):                 # plonk.create_proof's order: A' rows, S' rows, then the two blinds, lookup by lookup
            a_rows = [rand() for _ in range(bf + 1)]
            s_rows = [rand() for _ in range(bf + 1)]
            draws.append((a_rows, s_rows, rand(), rand()))
        per, lo, hi = parallel.block_range(L, self.world, self.rank)
        perm = self.torch.empty((max(per * self.world, 1), 2, self.n, 4), dtype=self.torch.int64, device="cuda")
        out, failure = [], None
        for li, (inputs, tables) in enumerate(lookups):
            d = {"pi": perm[li, 0], "pt": perm[li, 1], "pi_blind": draws[li][2], "pt_blind": draws[li][3], "ci": None, "ct": None}
            if lo <= li < hi and failure is None:
                try:
                    d["ci"], d["ct"] = self.compress(inputs, theta, values_of), self.compress(tables, theta, values_of)
                    pi, pt = self.permute_expression_pair(d["ci"], d["ct"], usable)
                except ValueError as e:                       # ConstraintSystemFailure: an input value absent from the table
                    failure = e
                    continue
                self.set_rows(pi, usable, draws[li][0])
                self.set_rows(pt, usable, draws[li][1])
                perm[li, 0].copy_(pi); perm[li, 1].copy_(pt)
            out.append(d)
        if self.world > 1 and L:
            # a failed lookup is seen by its owner only: agree on the outcome before anybody enters the bulk collective
            ok = self.torch.tensor([0 if failure is not None else 1], dtype=self.torch.int32, device="cuda")
            self.dist.all_reduce(ok, op=self.dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                from .lookup import ConstraintSystemFailure
                raise failure if failure is not None else ConstraintSystemFailure("lookup input value not present in the table (on another rank)")
            parallel.all_gather_blocks_inplace(perm, per, self.dist)
        elif failure is not None:
            raise failure
        return out

    def lookup_products(self, lookups, beta, gamma, bf, rand):
        L = len(lookups)
        draws = []
        for _ in range(L):
            rows = [rand() for _ in range(bf)]
            draws.append((rows, rand()))
        per, lo, hi = parallel.block_range(L, self.world, self.rank)
        zs = self.torch.empty((max(per * self.world, 1), self.n, 4), dtype=self.torch.int64, device="cuda")
        for li, d in enumerate(lookups):
            if lo <= li < hi:
                self.ctx.check(self.lib.trp_dev_lookup_product(self.dom.handle, d["ci"].data_ptr(), d["ct"].data_ptr(), d["pi"].data_ptr(),
                                                               d["pt"].data_ptr(), self._m(beta), self._m(gamma), zs[li].data_ptr(), self.n - bf))
                self.set_rows(zs[li], self.n - bf, draws[li][0])
            d["z"], d["z_blind"] = zs[li], draws[li][1]
        if self.world > 1 and L:
            parallel.all_gather_blocks_inplace(zs, per, self.dist)

    # -- permutation argument: chunks from 1, scaled by the product of their predecessors' ends ---------------------------------------------
    def permutation_commit(self, values, sigmas, beta, gamma, chunk_len, blinding_factors, rand, after_chunk):
        if self.world == 1:
            return super().permutation_commit(values, sigmas, beta, gamma, chunk_len, blinding_factors, rand, after_chunk)
        from ._lib import ptr
        n, p, ct, t, bf = self.n, self.p, self.ct, self.torch, blinding_factors
        starts = list(range(0, len(values), chunk_len))
        C = len(starts)
        per, lo, hi = parallel.block_range(C, self.world, self.rank)
        zs = t.empty((per * self.world, n, 4), dtype=t.int64, device="cuda")
        rows = []
        for ci in range(C):                # halo2's draw order: a chunk's blinding rows, then (after_chunk) its blind
            rows.append([rand() for _ in range(bf)])
            after_chunk(zs[ci])
        u = n - (bf + 1)
        ends = t.zeros((per * self.world, 4), dtype=t.int64, device="cuda")
        for ci in range(lo, hi):
            cols = list(range(starts[ci], min(starts[ci] + chunk_len, len(values))))
            dbeta = self._limbs([pow(self.delta, c, p) * beta % p for c in cols])
            vptr = (ct.c_void_p * len(cols))(*[values[c].data_ptr() for c in cols])
            sptr = (ct.c_void_p * len(cols))(*[sigmas[c].data_ptr() for c in cols])
            self.ctx.check(self.lib.trp_dev_permutation_product(self.dom.handle, vptr, sptr, len(cols), self._m(beta), self._m(gamma), ptr(dbeta),
                                                                None, zs[ci].data_ptr()))
            ends[ci].copy_(zs[ci][u])
        parallel.all_gather_blocks_inplace(ends, per, self.dist)
        pref = parallel.chunk_prefixes(self._ints(ends[:C].cpu().numpy().view(self.np.uint64)), p)
        for ci in range(lo, hi):
            if pref[ci] != 1:
                d_s = self._dev(self._limbs([pref[ci]]))
                self.ctx.check(self.lib.trp_dev_field_op(self.ctx.handle, 0, 2 | 16, zs[ci].data_ptr(), d_s.data_ptr(), zs[ci].data_ptr(), u + 1))
            self.set_rows(zs[ci], n - bf, rows[ci])
        parallel.all_gather_blocks_inplace(zs, per, self.dist)
        return [zs[ci] for ci in range(C)]

    # -- key material: each rank keeps its ROW SLICE (with halo) of the j - 1 cosets -------------------------------------------------------
    def _slice_rows(self):
        row0, S = parallel.row_slice_bounds(self.n, self.world, self.rank)
        t = self.torch
        idx = (t.arange(S + 2 * self.HALO, device="cuda") + (row0 - self.HALO)) % self.n
        return row0, S, idx

    def coeff_to_extended_static(self, c):
        if self.world == 1:
            return super().coeff_to_extended_static(c)
        ncos = self.j - 1
        row0, S, idx = self._slice_rows()
        held = sum(v.numel() for v in self._static.values()) * 8
        if held + ncos * (S + 2 * self.HALO) * 32 > self.static_budget_bytes:
            return c
        full = self._buf("static_full", (self.n, 4))
        vals = self.torch.empty((ncos, S + 2 * self.HALO, 4), dtype=self.torch.int64, device="cuda")
        for cs in range(ncos):
            self.ctx.check(self.lib.trp_dev_coeff_to_coset(self.dom.handle, c.data_ptr(), full.data_ptr(), 1, cs))
            vals[cs] = full[idx]
        self._static[id(c)] = vals
        self._static_keep.append(c)
        return c

    # -- the quotient: NTTs by column block, program by row slice --------------------------------------------------------------------------
    def quotient_pieces(self, pk, challenges, build_h, build_parts, resolve):
        """one GPU: GpuBackend's (the numerator split by constraint degree); several: the whole program, row-sliced by quotient()"""
        if self.world == 1:
            return super().quotient_pieces(pk, challenges, build_h, build_parts, resolve)
        cached = self.quotient_program(pk, build_h, challenges, len(pk.vk.cs.permutation))
        prog, keys = cached if cached is not None else build_h(*challenges)
        return self.quotient(prog, [resolve(k_) for k_ in keys])

    def quotient(self, ast, ext_polys):
        self._drain()
        t, n, ncos, G, H = self.torch, self.n, self.j - 1, self.world, self.HALO
        dyn = [i for i, c in enumerate(ext_polys) if id(c) not in self._static]
        in_arena = [self._arena_slot.get(id(ext_polys[i])) for i in dyn]
        if dyn and all(a is not None and a[1] is ext_polys[i] for a, i in zip(in_arena, dyn)):
            coeff = self._arena[:self._arena_used]
            slot = {i: a[0] for a, i in zip(in_arena, dyn)}
        else:
            coeff = t.stack([ext_polys[i] for i in dyn]) if dyn else t.empty((0, n, 4), dtype=t.int64, device="cuda")
            slot = {i: s_ for s_, i in enumerate(dyn)}
        ncols = coeff.shape[0]
        per, lo, hi = parallel.block_range(ncols, G, self.rank)
        row0, S, _ = self._slice_rows()
        width = S + 2 * H
        own = self._buf("q_own", (max(per, 1), n, 4))
        send = [self._buf(f"q_send{b}", (G, max(per, 1), width, 4)) for b in (0, 1)]
        recv = [self._buf(f"q_recv{b}", (G, max(per, 1), width, 4)) for b in (0, 1)]
        local = t.empty((ncos, S, 4), dtype=t.int64, device="cuda")
        prog = None

        def run_program(cs, handle):
            if handle is not None:
                handle.wait()                              # the prover's stream waits for the exchange of this coset
            flat = recv[cs & 1].view(G * max(per, 1), width, 4)
            ptrs = [flat[slot[i]].data_ptr() if i in slot else self._static[id(c)][cs].data_ptr() for i, c in enumerate(ext_polys)]
            self.ev.evaluate_device_rows(prog, self.dom, ptrs, local[cs].data_ptr(), cs, row0, S, H, H)

        # software pipeline over the cosets: the all-to-all of coset c runs on NCCL's stream while this rank's NTTs of coset c + 1
        # run on the prover's stream; the program of coset c follows.  The program is compiled (host) while the first NTTs run.
        pending = None
        for cs in range(ncos):
            if hi > lo:
                self.ctx.check(self.lib.trp_dev_coeff_to_coset(self.dom.handle, coeff[lo].data_ptr(), own.data_ptr(), hi - lo, cs))
                parallel.pack_row_slices(own, hi - lo, n, G, H, H, send[cs & 1])
            handle = self.dist.all_to_all_single(recv[cs & 1], send[cs & 1], async_op=True) if ncols else None
            if prog is None:
                prog = ast if isinstance(ast, P.Program) else P.compile_ast(ast, self.p)
            if pending is not None:
                run_program(*pending)
            pending = (cs, handle)
        run_program(*pending)
        gathered = t.empty((G, ncos, S, 4), dtype=t.int64, device="cuda")
        self.dist.all_gather_into_tensor(gathered, local)
        vals = gathered.permute(1, 0, 2, 3).reshape(ncos, n, 4).contiguous()
        h = t.empty((ncos, n, 4), dtype=t.int64, device="cuda")
        self.ctx.check(self.lib.trp_dev_cosets_to_coeff(self.dom.handle, vals.data_ptr(), ncos, h.data_ptr(), 1))
        return [h[i] for i in range(ncos)]
