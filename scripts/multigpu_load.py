"""Multi-rank check of wafer_load_array (run under torchrun, one rank per GPU): files written by a single-GPU context
(a seeded Gaussian psi and a Harmonic V of a coarser lattice) are loaded by every rank of an x-slab decomposed lattice
as psi, V and a lower state; the slab checksums, added over the ranks, must equal those of a single-GPU context that
loads the same files, and the multi-rank V must write the same file.  Rank 0 prints one JSON line; exit code 1 on a
mismatch."""
import json
import os
import shutil
import sys
import tempfile

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

    def total(lat):
        s, x = lat.phi_checksum()
        t = torch.tensor([s & 0xFFFFFFFF, s >> 32, x & 0xFFFFFFFF, x >> 32], dtype=torch.int64, device="cuda")
        parts = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(parts, t)
        s_all, x_all = 0, 0
        for p in parts:
            p = [int(v) for v in p.tolist()]
            s_all = (s_all + (p[0] | p[1] << 32)) & (2 ** 64 - 1)
            x_all ^= p[2] | p[3] << 32
        return s_all, x_all

    box = [tempfile.mkdtemp(prefix="wafer_load_") if rank == 0 else None]
    dist.broadcast_object_list(box, 0)
    d = box[0]
    results, ok = {}, True
    kw = dict(dn=0.1, dt=2e-3, mass=1.0, device=local)
    for cd, shape, src in (("ThreePoint", (96, 41, 72), (50, 30, 33)), ("FivePoint", (50, 33, 40), (50, 33, 40)),
                           ("SevenPoint", (41, 24, 31), (70, 20, 45))):
        if rank == 0:  # the input files
            with wafer_b200.Lattice(src, cd, **kw) as w:
                w.generate_potential("Harmonic")
                w.set_initial_conditions("Gaussian", sig=1.3, seed=0x5EED0000CAFE)
                for ft, ext in ((0, ".mpk"), (1, ".csv"), (2, ".json")):
                    w.write_array("phi", os.path.join(d, "%s_phi%s" % (cd, ext)), ft)
                    w.write_array("potential", os.path.join(d, "%s_v%s" % (cd, ext)), ft)
        dist.barrier()
        for ft, ext in ((0, ".mpk"), (1, ".csv"), (2, ".json")):
            fphi, fv = os.path.join(d, "%s_phi%s" % (cd, ext)), os.path.join(d, "%s_v%s" % (cd, ext))
            sums = {}
            for name, w_, r_ in (("single", 1, 0), ("multi", world, rank)):
                if name == "single" and rank != 0:
                    lat = None
                else:
                    lat = wafer_b200.Lattice(shape, cd, rank=r_, world=w_,
                                             nccl_id=fresh_nccl_id() if w_ > 1 else None, **kw)
                if name == "single":
                    dist.barrier()
                    if lat is None:
                        continue
                lat.load_array("potential", fv, ft)
                lat.load_array("lower", fphi, ft)
                lat.load_array("phi", fphi, ft)
                tot = total(lat) if w_ > 1 else lat.phi_checksum()
                lat.phi_from_lower(0)
                tot_lower = total(lat) if w_ > 1 else lat.phi_checksum()
                vpath = os.path.join(d, "%s_v_%s%s" % (cd, name, ext))
                lat.write_array("potential", vpath, ft)
                sums[name] = (tot, tot_lower, vpath)
                lat.close()
            if rank == 0:
                (a, al, ap), (b, bl, bp) = sums["single"], sums["multi"]
                with open(ap, "rb") as fa, open(bp, "rb") as fb:
                    same_v = fa.read() == fb.read()
                res = a == b and al == bl and same_v
                results["%s%s" % (cd, ext)] = res
                ok = ok and res
            dist.barrier()
    if rank == 0:
        shutil.rmtree(d, ignore_errors=True)
        print(json.dumps({"world": world, "ok": ok, "results": results}), flush=True)
    flag = torch.tensor([0 if ok else 1], device="cuda")
    dist.broadcast(flag, 0)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(int(flag.item()))


if __name__ == "__main__":
    main()
