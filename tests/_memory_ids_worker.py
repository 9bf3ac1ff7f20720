"""Worker of tests/test_gpu_memory_ids.py: launched by torchrun with >= 2 GPUs (NCCL).  Each rank owns a region memory
holding its own previous step's rows, tagged with its triplets' ids, and passes its own query ids: the fused step's
InfoNCE and logit-scale gradient on each rank equal the rank-local oracle (this rank's queries against every rank's
regions plus this rank's memory rows whose id is not the query's), over the peer exchange and over the NCCL collectives
(COR_PEER=0)."""
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
    qids = torch.arange(B, device=dev) + 10 * rank        # rank-local ids; rank r's ids also tag rows of rank r's memory only
    for use_peer in ("1", "0"):
        os.environ["COR_PEER"] = use_peer
        mem = region.RegionMemory(K, C, dev)
        mem.enqueue(torch.nn.functional.normalize(torch.randn(600 + 50 * rank, C, device=dev, generator=g), dim=-1),
                    ids=torch.randint(-1, 10 * ws, (600 + 50 * rank,), device=dev, generator=g))
        steps = []
        for i in range(2):                                  # the second step finds the first step's rows in the memory
            s = torch.tensor(9.0, dtype=torch.float32, device=dev, requires_grad=True)
            p, e, c = (t[k].clone().requires_grad_(True) for k in ("pred", "emb", "comb"))
            rows_before, ids_before = mem.rows(), mem.row_ids()
            out = region.region_step(p, e, c, t["masks"], fused=True, logit_scale=s, nce_weight=1.3, memory=mem, query_ids=qids)
            out.loss.backward(torch.tensor(0.7, device=dev))
            rows = out.regions.reshape(B * M, C).contiguous()
            allr = [torch.empty_like(rows) for _ in range(ws)]
            dist.all_gather(allr, rows)
            R = torch.cat(allr).bfloat16().double().cpu()
            Q = t["comb"].reshape(B, C).bfloat16().double().cpu()
            st = torch.tensor(9.0, dtype=torch.float64, requires_grad=True)
            logits = st * (Q @ torch.cat([R, rows_before.double().cpu()]).t())
            mi, qi = ids_before.cpu(), qids.cpu()
            excl = (mi[None, :] >= 0) & (mi[None, :] == qi[:, None])
            keep = torch.cat([torch.ones(B, R.shape[0], dtype=torch.bool), ~excl], 1)
            logits = logits.masked_fill(~keep, float("-inf"))
            tg = torch.arange(B) * M + rank * B * M
            nce = (torch.logsumexp(logits, 1) - logits[torch.arange(B), tg]).mean()
            (0.7 * 1.3 * nce).backward()
            assert abs(float(out.nce) - float(nce)) <= 1e-3 * abs(float(nce)), f"COR_PEER={use_peer} rank {rank} step {i}: nce"
            got, ref = float(s.grad), float(st.grad)
            assert abs(got - ref) <= 1e-3 * abs(ref), f"COR_PEER={use_peer} rank {rank} step {i}: {got} vs {ref}"
            mem.enqueue(out.regions, ids=qids)
            steps.append(int(excl.sum()))
        assert steps[1] > steps[0], f"rank {rank}: the second step excludes the first step's own rows"
    torch.cuda.synchronize()
    dist.barrier()
    if rank == 0:
        print("MEMORY_IDS_OK", ws, flush=True)
    peer.release_all()
    os._exit(0)


if __name__ == "__main__":
    main()
