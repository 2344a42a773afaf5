"""Host logic of the Ulysses context-parallel path (SURVEY.md N2) without GPUs: the ownership plan (rows, heads, rank-major
joint order, destination-major QKV weight rows) is exercised by a world_size-2 `gloo` emulation of exactly the data movement
the kernels perform on B200s - destination d receives [q | k | v] columns of its heads from every rank's rows, attends over the
whole (rank-major) sequence, and every output row returns to the rank that owns it - and must reproduce unsharded joint
attention.  The GPU version of the same statement is tests/multi_gpu_flux_cp.py."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from diffusers_b200.context_parallel import ContextParallelConfig, UlyssesPlan


def test_plan_partitions_rows_and_heads():
    for world in (2, 4, 8):
        plans = [UlyssesPlan(world, r, 512, 4096, 24, 128) for r in range(world)]
        p = plans[0]
        assert p.L == 4608 and p.Ll * world == p.L and p.hl * world == 24 and p.Dl * world == p.D == 3072
        g = p.joint_to_rank_major()
        assert sorted(g.tolist()) == list(range(p.L))  # a permutation of the joint sequence
        for r, q in enumerate(plans):
            b0, b1 = q.block()
            t0, t1 = q.text_rows()
            s0, s1 = q.image_rows()
            assert g[b0:b0 + q.Tl].tolist() == list(range(t0, t1))
            assert g[b0 + q.Tl:b1].tolist() == list(range(q.T + s0, q.T + s1))
            assert sorted(q.send_order()) == list(range(world)) and q.send_order()[-1] == r
        perm = p.qkv_row_permutation()
        assert sorted(perm.tolist()) == list(range(3 * p.D))
        for d in range(world):
            rows = perm[d * 3 * p.Dl:(d + 1) * 3 * p.Dl]
            assert rows[:p.Dl].tolist() == list(range(d * p.Dl, (d + 1) * p.Dl))                      # q of d's heads
            assert rows[p.Dl:2 * p.Dl].tolist() == list(range(p.D + d * p.Dl, p.D + (d + 1) * p.Dl))  # k
            assert rows[2 * p.Dl:].tolist() == list(range(2 * p.D + d * p.Dl, 2 * p.D + (d + 1) * p.Dl))  # v


def test_plan_and_config_refuse_what_is_not_built():
    with pytest.raises(ValueError):
        UlyssesPlan(2, 0, 24, 64, 3, 64)       # heads % world
    with pytest.raises(ValueError):
        UlyssesPlan(2, 0, 24, 64, 2, 64)       # 12 text rows per rank: not 16-byte-row aligned slices of 8
    with pytest.raises(NotImplementedError):
        ContextParallelConfig(ring_degree=2)
    with pytest.raises(NotImplementedError):
        ContextParallelConfig(ulysses_degree=2, ulysses_anything=True)
    assert ContextParallelConfig(ulysses_degree=4).ring_degree == 1


def _exchange(send, rank, world):
    """all-to-all of equal-sized pieces (gloo has no alltoall: every rank gathers all send lists and keeps its column)."""
    mine = torch.stack(send)
    everyone = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(everyone, mine)
    return [everyone[s][rank] for s in range(world)]


def _attend(q, k, v, heads, hd):
    L = q.shape[0]
    qh, kh, vh = (t.view(L, heads, hd).transpose(0, 1) for t in (q, k, v))
    return torch.nn.functional.scaled_dot_product_attention(qh, kh, vh).transpose(0, 1).reshape(L, heads * hd)


def _worker(rank, world, port, q_out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        T, S, heads, hd, Dm = 16, 48, 4, 8, 24
        plan = UlyssesPlan(world, rank, T, S, heads, hd)
        D, Dl, Ll, L = plan.D, plan.Dl, plan.Ll, plan.L
        g = torch.Generator().manual_seed(5)
        x = torch.randn(L, Dm, generator=g, dtype=torch.float64)          # joint order [text | image]
        W = torch.randn(3 * D, Dm, generator=g, dtype=torch.float64)
        pos = torch.rand(L, 1, generator=g, dtype=torch.float64) + 0.5    # stand-in for the position-dependent rotary factor
        qkv = x @ W.T
        ref = _attend(qkv[:, :D] * pos, qkv[:, D:2 * D] * pos, qkv[:, 2 * D:], heads, hd)

        # ---- what rank `rank` does
        (t0, t1), (s0, s1) = plan.text_rows(), plan.image_rows()
        x_loc = torch.cat([x[t0:t1], x[T + s0:T + s1]])                   # [its text | its image]
        y = x_loc @ W[plan.qkv_row_permutation()].T                        # [Ll, 3D], destination-major columns
        send = [y[:, d * 3 * Dl:(d + 1) * 3 * Dl].contiguous() for d in range(world)]
        recv = _exchange(send, rank, world)                                # (the GEMM epilogue's peer stores)
        J = torch.cat(recv)                                                # rank-major rows: sender s at [s*Ll, (s+1)*Ll)
        pos_rm = pos[plan.joint_to_rank_major()]
        o = _attend(J[:, :Dl] * pos_rm, J[:, Dl:2 * Dl] * pos_rm, J[:, 2 * Dl:], plan.hl, hd)   # my heads, whole sequence
        send = [o[s * Ll:(s + 1) * Ll].contiguous() for s in range(world)]  # rows go back to their owners
        recv = _exchange(send, rank, world)                                # (the attention epilogue's o_seg stores)
        A = torch.cat(recv, dim=1)                                         # columns [s*Dl, (s+1)*Dl) from rank s
        want = torch.cat([ref[t0:t1], ref[T + s0:T + s1]])
        err = float((A - want).abs().max())
        q_out.put((rank, "ok" if err < 1e-10 else f"max err {err}"))
    except Exception as e:  # noqa: BLE001
        q_out.put((rank, repr(e)))
    finally:
        dist.destroy_process_group()


def _enable_worker(rank, world, port, q_out):
    """FluxTransformer2DModel.enable_parallelism on the host (gloo, CPU buffers): the QKV weights / biases of every block end up in
    destination blocks in send order, the API refuses what is not built, and the permuted model no longer exports a checkpoint."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from diffusers_b200 import packing, specs
        from diffusers_b200.transformer_flux import FluxTransformer2DModel
        cfg = dict(patch_size=1, in_channels=16, num_layers=1, num_single_layers=1, attention_head_dim=64, num_attention_heads=4,
                   joint_attention_dim=32, pooled_projection_dim=16, guidance_embeds=True, axes_dims_rope=(8, 28, 28))
        sd = specs.random_state_dict(specs.flux_params(dict(specs.FLUX_DEV_CONFIG, **cfg)), seed=3)
        m = FluxTransformer2DModel(cfg, sd, device="cpu")
        for bad in (dict(ulysses_degree=4), dict(ulysses_degree=1)):
            try:
                m.enable_parallelism(config=ContextParallelConfig(**bad))
                raise AssertionError("a degree that differs from the group size must be refused")
            except ValueError:
                pass
        try:
            m.enable_parallelism(config=ContextParallelConfig(ulysses_degree=2), cp_plan={"": {}})
            raise AssertionError("custom cp_plan must be refused")
        except NotImplementedError:
            pass
        m.enable_parallelism(config=ContextParallelConfig(ulysses_degree=world))
        plan = UlyssesPlan(world, rank, 16, 16, 4, 64)
        D, Dl = plan.D, plan.Dl
        a = "transformer_blocks.0.attn"
        full_w = torch.cat([sd[a + ".to_q.weight"], sd[a + ".to_k.weight"], sd[a + ".to_v.weight"]], 0)
        full_b = torch.cat([sd[a + ".to_q.bias"], sd[a + ".to_k.bias"], sd[a + ".to_v.bias"]], 0)
        w = packing.unpack_linear_weight(m.W(m.double[0]["qkv"]["w"]).cpu(), D)
        b = m.W(m.double[0]["qkv"]["b"]).cpu()
        for i, d in enumerate(plan.send_order()):
            for part in range(3):  # block i = [q | k | v] rows of the heads rank d owns
                rows = slice(part * D + d * Dl, part * D + (d + 1) * Dl)
                blk = slice(i * 3 * Dl + part * Dl, i * 3 * Dl + (part + 1) * Dl)
                assert torch.equal(w[blk], full_w[rows]) and torch.equal(b[blk], full_b[rows]), (i, d, part)
        # the text-stream projection and the single blocks are permuted the same way; everything else is untouched
        aw = packing.unpack_linear_weight(m.W(m.double[0]["aqkv"]["w"]).cpu(), D)
        assert torch.equal(aw[:Dl], sd[a + ".add_q_proj.weight"][plan.send_order()[0] * Dl:(plan.send_order()[0] + 1) * Dl])
        assert torch.equal(packing.unpack_linear_weight(m.W(m.double[0]["out"]["w"]).cpu(), D), sd[a + ".to_out.0.weight"])
        for must_fail, exc in ((lambda: m.reference_state_dict(), RuntimeError),
                               (lambda: m.enable_parallelism(config=ContextParallelConfig(ulysses_degree=world)), RuntimeError)):
            try:
                must_fail()
                raise AssertionError("expected a refusal")
            except exc:
                pass
        q_out.put((rank, "ok"))
    except Exception as e:  # noqa: BLE001
        q_out.put((rank, repr(e)))
    finally:
        dist.destroy_process_group()


def _run_two(worker):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    return sorted(res)


def _peer_failure_worker(rank, world, port, q_out):
    """b200_peer_alloc fails on every rank: the failure must surface as the SAME error on all ranks (after the outcome
    exchange), not as one rank raising while the other waits in a collective."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import torch.cuda
        from diffusers_b200 import _lib
        from diffusers_b200 import context_parallel as cp
        real = _lib.lib()

        class NoPeerMemory:  # the allocation fails as it does without a device, whether or not this host has a GPU
            def __getattr__(self, name):
                return getattr(real, name)

            @staticmethod
            def b200_peer_alloc(nbytes, ptr, handle):
                return 1

            @staticmethod
            def b200_last_error():
                return b"no CUDA device"

        torch.cuda.current_device = lambda: 0      # host-only stand-ins: the allocation itself is what must fail
        _lib.init = lambda d: None
        _lib.lib = lambda: NoPeerMemory()
        try:
            cp.PeerBuffer(1 << 20)
            q_out.put((rank, "no error"))
        except cp.B200Error as e:
            q_out.put((rank, "ok" if "could not allocate the peer buffers on rank(s) [0, 1]" in str(e) else repr(e)))
    except Exception as e:  # noqa: BLE001
        q_out.put((rank, repr(e)))
    finally:
        dist.destroy_process_group()


def test_peer_buffer_failures_are_raised_on_every_rank():
    assert _run_two(_peer_failure_worker) == [(0, "ok"), (1, "ok")]


def test_enable_parallelism_host_side_two_rank_gloo():
    assert _run_two(_enable_worker) == [(0, "ok"), (1, "ok")]


def test_enable_parallelism_needs_an_initialized_process_group():
    from diffusers_b200 import specs
    from diffusers_b200.transformer_flux import FluxTransformer2DModel
    cfg = dict(patch_size=1, in_channels=16, num_layers=1, num_single_layers=1, attention_head_dim=64, num_attention_heads=2,
               joint_attention_dim=32, pooled_projection_dim=16, guidance_embeds=True, axes_dims_rope=(8, 28, 28))
    m = FluxTransformer2DModel(cfg, specs.random_state_dict(specs.flux_params(dict(specs.FLUX_DEV_CONFIG, **cfg)), seed=3), device="cpu")
    with pytest.raises(RuntimeError):
        m.enable_parallelism(config=ContextParallelConfig(ulysses_degree=2))
    with pytest.raises(NotImplementedError):
        m.enable_parallelism(config=object())


def test_two_rank_gloo_ulysses_data_movement_equals_joint_attention():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, "ok"), (1, "ok")], res
