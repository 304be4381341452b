"""The optimiser's data-parallel forms -- rlppo_norm_clip_adam_peers (one-shot: every rank sums all peers' gradient arenas
over NVLink) and rlppo_norm_clip_adam_peers2 (two-shot: every rank reduces its slice, then gathers the reduced slices) --
under torchrun, one rank per GPU:  python -m torch.distributed.run --standalone --nproc-per-node N tests/optim_peers_check.py

Every rank holds its gradient arena, flag block and (two-shot) reduced buffer in symmetric memory, as
PPOLearner._setup_peers does, and makes several consecutive launches per layout and form, rewriting its arena before each
one and starting it after a random per-rank delay.  After every launch:
  * the summed gradient (the one-shot form's `gsum`, the two-shot form's own reduced buffer) is the host fp32 sum of all
    ranks' gradients taken in rank order 0..R-1, bit for bit;
  * p, m, v, the step counts and the sums of squares are bit-identical to a one-rank rlppo_norm_clip_adam on that summed
    gradient from the same state (the kernel keeps the thread <-> element mapping, the accumulation order and the grid of
    the one-rank form in both peer forms);
  * where views are passed, the bf16 operands hold bf16 of the new weights;
and at the end every rank's snapshots are the same bits.
Layouts: the learner's 3-segment arena (metric tail at lr 0), totals 5 and 13 (two-shot slices of 4 leave ranks without
elements from world 3 up), a total that is not a multiple of 4 x world, and an arena above the one-shot size threshold."""
import os
import sys
import zlib

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LAUNCHES = 4
SENTINEL = -77.0


def layouts(world):
    from rlgym_ppo_b200 import parallel
    big = parallel.ONE_SHOT_BYTES // 4 + 12345          # above the one-shot threshold at every world size >= 2
    odd = 4 * world * 2500 + 2 * world + 1
    return {"dp": [0, 177754, 332635, 332643], "5": [0, 5], "13": [0, 6, 6, 13], "odd": [0, 4000, odd],
            "big": [0, big // 2, big]}


def rank_grads(name, rank, it, n):
    """fp32 gradients of `rank` for launch `it` -- any rank can regenerate any other rank's."""
    rng = np.random.default_rng([zlib.crc32(name.encode()), rank, it])
    return (rng.standard_normal(n, dtype=np.float32) * np.float32(1e-3 * (1 + rank))).astype(np.float32)


def bits(t):
    return t.contiguous().view(torch.int32) if t.element_size() == 4 else t.contiguous().view(torch.int16)


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    dist.init_process_group("nccl", device_id=dev)
    import torch.distributed._symmetric_memory as symm_mem
    from rlgym_ppo_b200 import _lib, ops

    lays = {k: np.asarray(v, np.int64) for k, v in layouts(world).items()}
    n_max = max(int(s[-1]) for s in lays.values())

    def symm(n, dtype):
        t = symm_mem.empty(n, dtype=dtype, device=dev)
        t.zero_()
        return t, [int(x) for x in symm_mem.rendezvous(t, dist.group.WORLD).buffer_ptrs]

    grads, grad_ptrs = symm(n_max, torch.float32)
    red, red_ptrs = symm(n_max, torch.float32)
    flags, flag_ptrs = symm(int(_lib._lib.rlppo_peer_flag_bytes()) // 4, torch.int32)
    gsum = torch.zeros(n_max, dtype=torch.float32, device=dev)
    torch.cuda.synchronize()
    dist.barrier()
    delay = np.random.RandomState(99 + 7 * rank)
    errors = []

    def check(ok, msg):
        # failures are collected, not raised: a rank that stopped launching would leave its peers' kernels waiting
        if not ok:
            errors.append(msg)

    for name, seg in lays.items():
        n, k = int(seg[-1]), len(seg) - 1
        own = [torch.from_numpy(rank_grads(name, rank, it, n)).to(dev) for it in range(LAUNCHES)]
        for form in ("one_shot", "two_shot"):
            rng = np.random.default_rng(5)                  # the same initial state on every rank
            p = torch.from_numpy((rng.standard_normal(n) * 0.05).astype(np.float32)).to(dev)
            m = torch.from_numpy((rng.standard_normal(n) * 1e-3).astype(np.float32)).to(dev)
            v = torch.from_numpy((rng.random(n) * 1e-6).astype(np.float32)).to(dev)
            steps = torch.tensor([(0, 1, 7)[j % 3] for j in range(k)], dtype=torch.int64, device=dev)
            lr = torch.tensor([3e-4 / (1 + j) for j in range(k)], dtype=torch.float32, device=dev)
            if k == 3:
                lr[2] = 0.0
            sq = torch.zeros(k, dtype=torch.float32, device=dev)
            views, bufs = None, []
            if name == "dp":          # a 256 x 89 and an 89 x 300 weight, W and W^T with padded leading dimensions
                views = []
                for off, out_f, in_f in ((0, 256, 89), (177754, 89, 300)):
                    wq = torch.full((ops.pad8(out_f), ops.pad8(in_f)), SENTINEL, dtype=torch.bfloat16, device=dev)
                    wt = torch.full((ops.pad8(in_f), ops.pad8(out_f)), SENTINEL, dtype=torch.bfloat16, device=dev)
                    vw = _lib.Bf16View()
                    vw.offset, vw.out_f, vw.in_f = off, out_f, in_f
                    vw.wq, vw.wq_ld, vw.wt, vw.wt_ld = wq.data_ptr(), wq.stride(0), wt.data_ptr(), wt.stride(0)
                    views.append(vw)
                    bufs.append((off, out_f, in_f, wq, wt))
                views = (_lib.Bf16View * 2)(*views)
            snaps = []
            for it in range(LAUNCHES):
                grads[:n].copy_(own[it])
                if delay.rand() < 0.7:
                    torch.cuda._sleep(int(delay.randint(0, 400000)))      # up to ~0.2 ms of skew, per rank, per launch
                pre = [p.clone(), m.clone(), v.clone(), steps.clone(), lr.clone()]
                if form == "one_shot":
                    ops.norm_clip_adam_peers(p, grad_ptrs, flag_ptrs, rank, gsum, m, v, seg, sq, lr, steps, views=views)
                    summed = gsum[:n].clone()
                else:
                    ops.norm_clip_adam_peers2(p, grad_ptrs, flag_ptrs, red_ptrs, rank, m, v, seg, sq, lr, steps,
                                              views=views)
                    summed = red[:n].clone()
                post = [p.clone(), m.clone(), v.clone(), steps.clone(), sq.clone()]
                ops_views = [(b[0], b[1], b[2], b[3].clone(), b[4].clone()) for b in bufs]
                snaps.append((pre, post, summed, ops_views))
                lr.mul_(1.5)
            torch.cuda.synchronize()
            for it, (pre, post, summed, op_views) in enumerate(snaps):
                where = f"{name} {form} launch {it} rank {rank}/{world}"
                want = rank_grads(name, 0, it, n)
                for r in range(1, world):
                    want = want + rank_grads(name, r, it, n)        # fp32, rank order
                check(np.array_equal(summed.cpu().numpy().view(np.int32), want.view(np.int32)),
                      f"{where}: summed gradient differs from the rank-order fp32 sum")
                rp, rm, rv, rs, rl = (t.clone() for t in pre)
                rsq = torch.zeros(k, dtype=torch.float32, device=dev)
                ops.norm_clip_adam(rp, torch.from_numpy(want).to(dev), rm, rv, seg, rsq, rl, rs)
                for what, a, b in zip(("p", "m", "v", "steps", "sqnorm"), post, (rp, rm, rv, rs, rsq)):
                    check(torch.equal(bits(a), bits(b)), f"{where}: {what} differs from the one-rank launch")
                for off, out_f, in_f, wq, wt in op_views:
                    w = post[0][off:off + out_f * in_f].view(out_f, in_f).to(torch.bfloat16)
                    ref_q = torch.full_like(wq, SENTINEL)
                    ref_q[:out_f, :in_f] = w
                    ref_t = torch.full_like(wt, SENTINEL)
                    ref_t[:in_f, :out_f] = w.t()
                    check(torch.equal(bits(wq), bits(ref_q)) and torch.equal(bits(wt), bits(ref_t)),
                          f"{where}: bf16 operands of the {out_f} x {in_f} view are stale")
            mine = torch.cat([bits(t).view(torch.uint8).flatten() for _, post, _, _ in snaps for t in post])
            every = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(every, mine)
            check(all(torch.equal(e, every[0]) for e in every[1:]), f"{name} {form}: ranks hold different bits")
        dist.barrier()
    torch.cuda.synchronize()
    n_err = torch.tensor([len(errors)], device=dev)
    dist.all_reduce(n_err)
    for msg in errors[:10]:
        print(msg, flush=True)
    if int(n_err.item()) == 0 and rank == 0:
        print(f"optim_peers_check OK world={world} layouts={list(lays)} launches={LAUNCHES}", flush=True)
    dist.destroy_process_group()
    sys.exit(1 if int(n_err.item()) else 0)


if __name__ == "__main__":
    main()
