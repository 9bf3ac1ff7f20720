"""Worker of tests/test_gpu_logit_scale.py: launched by torchrun with >= 2 GPUs (NCCL).  The fused step's logit-scale
gradient on each rank equals the rank-local oracle -- the mean over the rank's own queries against every rank's
regions -- over the peer exchange and over the NCCL collectives (COR_PEER=0)."""
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
    from oracle import aten_port as ap

    B, M, C = 4, 16, 128
    d = synth.make_triplets(21 + rank, B=B, M=M, C=C, h=16, w=16, H=128, W=128, hp=32, wp=32, degenerate=False)
    t = {k: torch.from_numpy(v).to(dev) for k, v in d.items()}
    t["emb"] = t["emb"].bfloat16()
    assert region._fused_ok(t["emb"], t["masks"], "auto")
    for use_peer in ("1", "0"):
        os.environ["COR_PEER"] = use_peer
        s = torch.tensor(9.0, dtype=torch.float32, device=dev, requires_grad=True)
        p, e, c = (t[k].clone().requires_grad_(True) for k in ("pred", "emb", "comb"))
        out = region.region_step(p, e, c, t["masks"], fused=True, logit_scale=s, nce_weight=1.3)
        out.loss.backward(torch.tensor(0.7, device=dev))
        rows = out.regions.reshape(B * M, C).contiguous()
        allr = [torch.empty_like(rows) for _ in range(ws)]
        dist.all_gather(allr, rows)
        R = torch.cat(allr).double().cpu()
        st = torch.tensor(9.0, dtype=torch.float64, requires_grad=True)
        nce = ap.infonce(R, t["comb"].reshape(B, C).double().cpu(), torch.arange(B) * M + rank * B * M, tau=1.0 / st)
        (0.7 * 1.3 * nce).backward()
        got, ref = float(s.grad), float(st.grad)
        assert abs(got - ref) <= 1e-3 * abs(ref), f"COR_PEER={use_peer} rank {rank}: {got} vs {ref}"
    torch.cuda.synchronize()
    dist.barrier()
    if rank == 0:
        print("LOGIT_SCALE_OK", ws, flush=True)
    peer.release_all()
    os._exit(0)


if __name__ == "__main__":
    main()
