"""The two host->device wires of the proposal masks on one GPU: bounding-box crops (cim_mask_unpack_crops_tiled_meta_sparse)
against COCO compressed RLE strings (cim_mask_unpack_rle_tiled_meta_sparse), alternated over the same seeded batches.

Per workload shape (cfg2: 8 x 2000 masks of 512 x 512, cfg4: 8 x 2000 of 128 x 128; the bench's synthetic proposals,
seeds 1234 + b and 5234 + b for a second batch) it reports
  - the mask bytes per step of each wire;
  - the decode kernel against the sparse crop unpack: CUDA events around --calls launches that alternate the two
    batches (every call is a real sparse update), per round;
  - CIMHeadStep.run_host ms per step with either wire at prefetch depth 1 and 2 (lag_results, as bench.py's e2e),
    per round, the wires and depths alternated within each round.
The card's name and power limit are read in the same run.  One process, one GPU: the multi-rank effect (eight ranks
copying at once) is not measured here.

    python tools/rle_wire_bench.py [--rounds 5] [--calls 20] [--steps 10] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cim_b200 import _lib, heads, mask_ops, synth            # noqa: E402
from cim_b200.step import CIMHeadStep                        # noqa: E402

SHAPES = {"cfg2": dict(backbone="resnet50", n_img=8, R=2000, C=20, present=2, mask=512),
          "cfg4": dict(backbone="resnet50", n_img=8, R=2000, C=80, present=4, mask=128)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def batch(cfg, seed_base, dev):
    """one batch: rois, labels, both wires (host) and their device copies"""
    n_img, R, S = cfg["n_img"], cfg["R"], cfg["mask"]
    rois, labels, packed, flat = [], [], [], []
    for b in range(n_img):
        params = synth.proposal_params(R, 512, seed_base + b)
        rois.append(synth.rois_from_params(params, b))
        labels.append(synth.image_labels(cfg["C"], cfg["present"], seed_base + b))
        m = synth.rasterize(params, device=dev, out_size=S)
        packed.append(mask_ops.mask_pack(m, layout="tiled"))
        flat.append(mask_ops.mask_pack(m, layout="flat").cpu())
    packed = torch.stack(packed)
    crops = mask_ops.crops_from_packed_host(torch.stack(flat).view(n_img * R, -1), S, S)
    cnt = torch.full((n_img,), R, dtype=torch.int32, device=dev)
    idx = torch.arange(R, dtype=torch.int32, device=dev).repeat(n_img, 1).contiguous()
    chars, off, ln, _, _, need = mask_ops.mask_rle(packed, cnt, idx, S, S, kb_per_row=S // 16)
    assert int(need[0]) <= chars.numel() and int(need[1]) == 0
    rle = mask_ops.MaskRLE(chars[:int(need[0])].cpu(), off.view(-1).cpu(), ln.view(-1).cpu(),
                           torch.tensor([[S, S]] * n_img, dtype=torch.int32), S, S)
    d_crops = mask_ops.MaskCrops(crops.words.to(dev), crops.meta.to(dev), crops.off.to(dev), S, S)
    d_rle = mask_ops.MaskRLE(rle.chars.to(dev), rle.off.to(dev), rle.len.to(dev), rle.hw.to(dev), S, S)
    return dict(rois=torch.cat(rois), labels=torch.cat(labels), crops=crops, rle=rle, d_crops=d_crops, d_rle=d_rle,
                packed=packed)


def time_kernels(cfg, batches, calls, first, dev):
    """ms per sparse unpack call of each wire over the same alternating sequence of batches"""
    n_img, R, S = cfg["n_img"], cfg["R"], cfg["mask"]
    words = S * S // 32
    L = _lib.lib()
    st = _lib.stream_ptr(dev)
    out = {}
    for wire in (first, "rle" if first == "crops" else "crops"):
        packed = torch.zeros(n_img, R, words, dtype=torch.int32, device=dev)
        prev = torch.zeros(n_img * R, 4, dtype=torch.int32, device=dev)
        meta = torch.empty(L.cim_mask_meta_bytes(n_img, R, words), dtype=torch.uint8, device=dev)
        bad = torch.zeros(1, dtype=torch.int32, device=dev)

        def one(i):
            bt = batches[i % len(batches)]
            if wire == "rle":
                mask_ops._unpack_rle_into(bt["d_rle"], packed, prev, meta, bad, n_img, R, st)
            else:
                c = bt["d_crops"]
                _lib.check(L.cim_mask_unpack_crops_tiled_meta_sparse(
                    _lib.ptr(c.words), _lib.ptr(c.meta), _lib.ptr(c.off), _lib.ptr(packed), _lib.ptr(prev),
                    _lib.ptr(meta), meta.numel(), n_img, R, S, S, words, st), "crop unpack")

        for i in range(4):
            one(i)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(calls):
            one(i)
        e1.record()
        torch.cuda.synchronize()
        out[wire] = e0.elapsed_time(e1) / calls
        # both wires end on the same batch: same buffer
        out[wire + "_check"] = (packed.clone(), meta.clone())
    same = torch.equal(out["rle_check"][0], out["crops_check"][0])
    for w in ("rle_check", "crops_check"):
        del out[w]
    out["buffers_equal"] = bool(same)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--shapes", default="cfg2,cfg4")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    res = {"card": card(), "rounds": args.rounds, "kernel_calls": args.calls, "run_host_steps": args.steps,
           "multi_rank": "not measured (one process, one GPU)", "shapes": {}}
    for name in args.shapes.split(","):
        cfg = SHAPES[name]
        n_img, R, C, S = cfg["n_img"], cfg["R"], cfg["C"], cfg["mask"]
        batches = [batch(cfg, base, dev) for base in (1234, 5234)]
        r = {"mask_bytes_per_step": {"crops": int(np.mean([b["crops"].nbytes for b in batches])),
                                     "rle": int(np.mean([b["rle"].nbytes for b in batches]))},
             "longest_string": int(max(int(b["rle"].len.max()) for b in batches)),
             "kernel_ms": {"crops": [], "rle": []}, "buffers_equal": True,
             "run_host_ms": {f"depth{d}": {"crops": [], "rle": []} for d in (1, 2)}}
        r["bytes_ratio"] = r["mask_bytes_per_step"]["crops"] / r["mask_bytes_per_step"]["rle"]
        Cf, H, W, scale = synth.feature_shape(cfg["backbone"])
        gen = torch.Generator(device=dev).manual_seed(1234)
        feat = torch.randn(n_img, Cf, H, W, device=dev, generator=gen)
        grad_out = torch.randn(n_img * R, Cf, 7, 7, device=dev, generator=gen)
        seg_x = torch.randn(n_img * R, 4096, device=dev, generator=gen)
        torch.manual_seed(0)
        weight, bias = (t.detach().contiguous() for t in heads.cls_iou_model(4096, C + 1, 3).to(dev)._stacked())
        mat = torch.stack([synth.cluster_mat(R, C, (0, 1), 6, 1234 + b) for b in range(n_img)]).to(dev)
        steps = {}
        for d in (1, 2):
            for wire in ("crops", "rle"):
                st = CIMHeadStep(n_img, R, C, Cf, H, W, scale, S * S // 32, device=dev, mask_kb_per_row=S // 16,
                                 head_grads=True, order="graph")
                if wire == "crops":
                    cap = max(int(b["crops"].words.numel()) for b in batches) + 1024
                    st.alloc_host_io(mask_hw=(S, S), crop_capacity_words=cap, prefetch_depth=d)
                else:
                    cap = max(int(b["rle"].chars.numel()) for b in batches) + 1024
                    st.alloc_host_io(rle_capacity_bytes=cap, prefetch_depth=d)
                steps[(d, wire)] = st
        hp = torch.cuda.Stream(device=dev, priority=-1)

        def feed(st, wire, i):
            bt = batches[i % 2]
            st.wait_inputs_consumed()
            st.hi_rois.copy_(bt["rois"])
            st.hi_labels.copy_(bt["labels"])
            (st.set_host_crops(bt["crops"]) if wire == "crops" else st.set_host_rle(bt["rle"]))

        def run_host_ms(st, wire):
            np.random.seed(3)
            hp.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(hp):
                for i in range(3):
                    feed(st, wire, i)
                    st.run_host(feat, grad_out, seg_x, weight, bias, mat=mat, lag_results=True)
                st.flush_results()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(args.steps):
                    feed(st, wire, i + 3)
                    st.run_host(feat, grad_out, seg_x, weight, bias, mat=mat, lag_results=True)
                st.flush_results()
                e1.record()
                torch.cuda.synchronize()
            return e0.elapsed_time(e1) / args.steps, st.results_host

        for rnd in range(args.rounds):
            first = "crops" if rnd % 2 == 0 else "rle"
            k = time_kernels(cfg, batches, args.calls, first, dev)
            r["buffers_equal"] &= k.pop("buffers_equal")
            for w in ("crops", "rle"):
                r["kernel_ms"][w].append(k[w])
            for d in (1, 2):
                outs = {}
                for wire in ((first, "rle" if first == "crops" else "crops")):
                    ms, outs[wire] = run_host_ms(steps[(d, wire)], wire)
                    r["run_host_ms"][f"depth{d}"][wire].append(ms)
                r["buffers_equal"] &= bool(np.array_equal(np.nan_to_num(outs["crops"]["losses"], nan=-7.0),
                                                          np.nan_to_num(outs["rle"]["losses"], nan=-7.0)))
        r["kernel_ms_median"] = {w: float(np.median(v)) for w, v in r["kernel_ms"].items()}
        r["run_host_ms_median"] = {d: {w: float(np.median(v)) for w, v in x.items()} for d, x in r["run_host_ms"].items()}
        res["shapes"][name] = r
        del steps, batches
        torch.cuda.empty_cache()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
