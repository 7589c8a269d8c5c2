"""Multi-rank check of wafer_write_array (run under torchrun, one rank per GPU): psi (a seeded Gaussian, the same at any
world size) and V of an x-slab decomposed lattice, written by all ranks into one file per format, must equal byte for
byte the file a single-GPU context of the same lattice writes.  Rank 0 prints one JSON line; exit code 1 on mismatch."""
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

    box = [tempfile.mkdtemp(prefix="wafer_output_") if rank == 0 else None]
    dist.broadcast_object_list(box, 0)
    d = box[0]
    results, ok = {}, True
    for cd, shape in (("ThreePoint", (96, 41, 72)), ("FivePoint", (50, 33, 40)), ("SevenPoint", (41, 24, 31))):
        kw = dict(dn=0.1, dt=2e-3, mass=1.0, device=local)
        single = wafer_b200.Lattice(shape, cd, **kw) if rank == 0 else None
        multi = wafer_b200.Lattice(shape, cd, rank=rank, world=world, nccl_id=fresh_nccl_id(), **kw)
        for lat in (single, multi):
            if lat is not None:
                lat.generate_potential("Harmonic")
                lat.set_initial_conditions("Gaussian", sig=1.3, seed=0x5EED0000CAFE)
        for what in ("phi", "potential"):
            for ft, ext in ((0, ".mpk"), (1, ".csv"), (2, ".json")):
                mp = os.path.join(d, "%s_%s_multi%s" % (cd, what, ext))
                st = multi.write_array(what, mp, ft)
                t = torch.tensor([st["bytes"]], dtype=torch.int64, device="cuda")
                dist.all_reduce(t)
                if rank == 0:
                    sp = os.path.join(d, "%s_%s_single%s" % (cd, what, ext))
                    single.write_array(what, sp, ft)
                    with open(mp, "rb") as a, open(sp, "rb") as b:
                        same = a.read() == b.read()
                    res = same and int(t.item()) == st["file_bytes"] == os.path.getsize(sp)
                    results["%s/%s%s" % (cd, what, ext)] = res
                    ok = ok and res
                dist.barrier()
        if single is not None:
            single.close()
        multi.close()
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
