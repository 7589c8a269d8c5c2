"""Multi-rank check of the device resample of input files (run under torchrun, one rank per GPU): every rank passes the
whole source array to wafer_set_phi_resampled / wafer_set_potential_resampled, then 9 ground-state sweeps run on an
x-slab decomposed lattice; the start and the evolved field must equal, bit for bit, those of a single-GPU run of the
same lattice.  Each rank computes its own planes (ghost planes included) from global indices, so no rank needs
another's data.  Rank 0 prints one JSON line; exit code 1 on mismatch."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist

    import wafer_b200

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def fresh_nccl_id():
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt = torch.tensor(list(wafer_b200.nccl_unique_id()), dtype=torch.uint8, device="cuda")
        dist.broadcast(idt, 0)
        return bytes(idt.cpu().tolist())

    results, ok = {}, True
    rng = np.random.default_rng(41)
    for cd, shape, src_shape, csv in (("ThreePoint", (96, 41, 72), (37, 20, 29), False),
                                      ("FivePoint", (50, 33, 40), (120, 70, 90), True),
                                      ("SevenPoint", (41, 24, 31), (41, 24, 31), True)):
        src = rng.normal(size=src_shape)
        pot = np.abs(rng.normal(size=src_shape))
        kw = dict(dn=0.1, dt=2e-3, mass=1.0, device=local)
        single = wafer_b200.Lattice(shape, cd, **kw)
        multi = wafer_b200.Lattice(shape, cd, rank=rank, world=world, nccl_id=fresh_nccl_id(), **kw)
        x0, x1 = multi.slab
        sums = []
        for lat in (single, multi):
            lat.set_potential_resampled(pot, from_csv=csv)
            lat.set_phi_resampled(src, from_csv=csv)
            start = lat.phi_checksum(x0, x1)
            lat.evolve(0, 9)
            sums.append((start, lat.phi_checksum(x0, x1)))
        # the union over the ranks: add the wrapping sums, xor the xors (64-bit words travel as 32-bit halves)
        words = [w for pair in sums for c in pair for v in c for w in (v & 0xFFFFFFFF, v >> 32)]
        t = torch.tensor(words, dtype=torch.int64, device="cuda")
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank = [[int(w) for w in a.cpu().tolist()] for a in allt]

        def union(idx):  # idx: 0 single start, 1 single evolved, 2 multi start, 3 multi evolved
            s, x = 0, 0
            for w in per_rank:
                s = (s + w[4 * idx] + (w[4 * idx + 1] << 32)) % 2 ** 64
                x ^= w[4 * idx + 2] + (w[4 * idx + 3] << 32)
            return s, x

        res = dict(start=union(0) == union(2), evolved=union(1) == union(3))
        results[cd] = res
        ok = ok and res["start"] and res["evolved"]
        single.close()
        multi.close()
    if rank == 0:
        print(json.dumps({"world": world, "ok": ok, "results": results}), flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
