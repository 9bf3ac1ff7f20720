"""Worker of tests/test_gpu_memory.py: launched by torchrun with >= 2 GPUs (NCCL).  Each rank owns a region memory and
scores it against its own queries only: the fused step's InfoNCE and logit-scale gradient on each rank equal the
rank-local oracle (this rank's queries against every rank's regions plus this rank's memory rows), over the peer
exchange and over the NCCL collectives (COR_PEER=0)."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    rank, ws, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(lr)
    dev = torch.device("cuda", lr)
    dist.init_process_group("nccl", device_id=dev)
    from cor_b200 import peer, region, synth

    B, M, C, K = 4, 16, 128, 1000
    d = synth.make_triplets(31 + rank, B=B, M=M, C=C, h=16, w=16, H=128, W=128, hp=32, wp=32, degenerate=False)
    t = {k: torch.from_numpy(v).to(dev) for k, v in d.items()}
    t["emb"] = t["emb"].bfloat16()
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    for use_peer in ("1", "0"):
        os.environ["COR_PEER"] = use_peer
        mem = region.RegionMemory(K, C, dev)
        mem.enqueue(torch.nn.functional.normalize(torch.randn(700 + 50 * rank, C, device=dev, generator=g), dim=-1))
        s = torch.tensor(9.0, dtype=torch.float32, device=dev, requires_grad=True)
        p, e, c = (t[k].clone().requires_grad_(True) for k in ("pred", "emb", "comb"))
        out = region.region_step(p, e, c, t["masks"], fused=True, logit_scale=s, nce_weight=1.3, memory=mem)
        out.loss.backward(torch.tensor(0.7, device=dev))
        rows = out.regions.reshape(B * M, C).contiguous()
        allr = [torch.empty_like(rows) for _ in range(ws)]
        dist.all_gather(allr, rows)
        R = torch.cat(allr).bfloat16().double().cpu()
        Q = t["comb"].reshape(B, C).bfloat16().double().cpu()
        st = torch.tensor(9.0, dtype=torch.float64, requires_grad=True)
        logits = st * (Q @ torch.cat([R, mem.rows().double().cpu()]).t())
        tg = torch.arange(B) * M + rank * B * M
        nce = (torch.logsumexp(logits, 1) - logits[torch.arange(B), tg]).mean()
        (0.7 * 1.3 * nce).backward()
        assert abs(float(out.nce) - float(nce)) <= 1e-3 * abs(float(nce)), f"COR_PEER={use_peer} rank {rank}: nce"
        got, ref = float(s.grad), float(st.grad)
        assert abs(got - ref) <= 1e-3 * abs(ref), f"COR_PEER={use_peer} rank {rank}: {got} vs {ref}"
        mem.enqueue(out.regions)
        assert mem.count() == min(K, 700 + 50 * rank + B * M)
    torch.cuda.synchronize()
    dist.barrier()
    if rank == 0:
        print("MEMORY_OK", ws, flush=True)
    peer.release_all()
    os._exit(0)


if __name__ == "__main__":
    main()
