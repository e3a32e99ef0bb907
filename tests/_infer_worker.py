"""One rank of the evaluation checks: a resnet_tiny trainer (stub transport on CPU, or a GPU rank) runs
FusedDataParallelTrainer.evaluate on this rank's own seeded shard; the rank also writes its reference counts, computed with the
module's own eval forward, so the caller can compare the all-reduced result with the sum of the per-rank references."""
import argparse
import json
import os
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from batch_shipyard_b200.models.resnet import resnet_tiny  # noqa: E402
from batch_shipyard_b200.ops import coll  # noqa: E402
from batch_shipyard_b200.parallel.ddp import FusedDataParallelTrainer  # noqa: E402


def reference_counts(model, x_u8, y, to_input):
    """count / summed loss / top-1 / top-5 of the module's own eval forward (fp32 copy of the model)."""
    with torch.no_grad():
        logits = model(to_input(x_u8)).float()
    top = logits.topk(5, dim=1).indices
    hit = top == y.view(-1, 1)
    return {"count": int(y.numel()), "loss": float(F.cross_entropy(logits, y, reduction="sum")), "top1": int(hit[:, 0].sum()),
            "top5": int(hit.any(dim=1).sum())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rank", type=int, required=True)
    ap.add_argument("--world", type=int, required=True)
    ap.add_argument("--session", required=True)
    ap.add_argument("--device", type=int, default=-1)
    ap.add_argument("--out", required=True, help="directory for the per-rank reference counts")
    ap.add_argument("--image", type=int, default=32)
    a = ap.parse_args()
    gpu = a.device >= 0
    if gpu:
        torch.cuda.set_device(a.device)
    torch.manual_seed(0)
    comm = coll.Communicator(a.rank, a.world, device=a.device if gpu else None, session=a.session, heap_bytes=256 << 20)
    model = resnet_tiny(10)
    tr = FusedDataParallelTrainer(model, comm, (8, 3, a.image, a.image), 10, lr=0.01, use_graph=gpu)
    g = torch.Generator().manual_seed(100 + a.rank)
    n = 20 + 4 * a.rank                                  # a short last batch on every rank
    x = torch.randint(0, 256, (n, a.image, a.image, 3), dtype=torch.uint8, generator=g)
    y = torch.randint(0, 10, (n,), generator=g)
    ev = tr.evaluate(x, y, batch=8)
    # reference: an fp32 copy of the module through its own eval forward, on the conversion training uses
    ref_model = resnet_tiny(10)
    ref_model.load_state_dict({k: v.detach().float().cpu() for k, v in model.state_dict().items()})
    ref_model.eval()
    if gpu:
        from batch_shipyard_b200.ops import fused
        dev = torch.device("cuda", a.device)
        ref_model = ref_model.to(dev)

        def to_input(xx):
            xs = torch.empty((xx.shape[0], a.image // 2 + 3, a.image // 2 + 3, 16), dtype=torch.bfloat16, device=dev)
            fused.u8_to_s2d_norm(xx.to(dev), xs)
            return xs.float().permute(0, 3, 1, 2)
        ref = reference_counts(ref_model, x, y.to(dev), to_input)
    else:
        ref = reference_counts(ref_model, x, y, lambda xx: (xx.float() / 255.0).permute(0, 3, 1, 2))
    with open(os.path.join(a.out, f"ref.rank{a.rank}.json"), "w") as f:
        json.dump(ref, f)
    print("EVAL " + json.dumps(ev))
    comm.check_status()
    comm.close()
    print(" OK")


if __name__ == "__main__":
    main()
