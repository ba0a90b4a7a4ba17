"""Command line of the path: same argument names as the reference's examples/main.py:315-330, plus
`--tau` as a list (every tau from one distance pass), honest `--supervised` (the reference's loop at
main.py:348 overrides the flag) and `--dataset synthetic` (MVTec and the DINO weights are not available
offline; a folder loader is out of scope -- inject data loaders through driver.make_category_data).

    python -m anomaly_clustering_b200.main --dataset synthetic --backbone_names wideresnet50 \
        --layers_to_extract_from layer2 layer3 --pretrain_embed_dimension 1024 --target_embed_dimension 1024 \
        --tau 0.5 1 2 --output_dir outputs

writes outputs/<dataset>/<backbone>/<mode>/<layers>_<Dp>_<D>_<tau>_<ratio>/matrix_alpha_X_<category>_<mode>.pickle
(the reference's layout) and prints NMI / ARI / F1 per category and tau like examples/test.py:221-224."""
from __future__ import annotations

import argparse
import os

import torch

from . import backbones, cluster, driver, io


def synthetic_category(n_img: int, n_classes: int, seed: int, size: int = 224):
    """A 'bottle-shaped' synthetic category (SURVEY.md section 8d): smooth radial base pattern + noise,
    class c > 0 plants one defect type (blob / scratch / texture patch) at a random position."""
    gen = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, size), torch.linspace(-1, 1, size), indexing="ij")
    r = (yy ** 2 + xx ** 2).sqrt()
    base = torch.stack([torch.cos(6 * r), torch.sin(4 * r), 1 - r]).unsqueeze(0)
    imgs = base + 0.15 * torch.randn(n_img, 3, size, size, generator=gen)
    labels = []
    for i in range(n_img):
        c = i % n_classes
        labels.append("good" if c == 0 else "defect%d" % c)
        if c == 0:
            continue
        y0 = int(torch.randint(20, size - 80, (1,), generator=gen))
        x0 = int(torch.randint(20, size - 80, (1,), generator=gen))
        if c % 3 == 1:
            imgs[i, :, y0:y0 + 40, x0:x0 + 40] += 1.5
        elif c % 3 == 2:
            imgs[i, :, y0:y0 + 4, x0:x0 + 70] -= 2.0
        else:
            imgs[i, :, y0:y0 + 50, x0:x0 + 50] += 0.8 * torch.randn(3, 50, 50, generator=gen)
    loader = [{"image": imgs[i:i + 1], "is_anomaly": torch.tensor([int(labels[i] != "good")]), "anomaly": [labels[i]]}
              for i in range(n_img)]
    return loader, labels


def write_cli_csv(save_path, layers, pretrain_dim, target_dim, supervised, taus, rows) -> str:
    """rows = [(category, tau, NMI, ARI, F1)] -> the reference's <layers>_<Dp>_<D>_tau_result.csv (test.py:246-325),
    one block per tau, with the size-unweighted row set the CLI has (no object/texture split for synthetic data)."""
    blocks = [(("%g" % t), [(c, n, a, f) for c, tt, n, a, f in rows if tt == t]) for t in taus]
    return io.write_result_csv(io.result_csv_path(save_path, layers, pretrain_dim, target_dim), supervised, blocks)


# --backbone_dtype: None keeps the fp32 backbone; a 16-bit run tags its backbone directory
BACKBONE_DTYPES = {"float32": None, "bfloat16": torch.bfloat16, "float16": torch.float16}
_DTYPE_TAGS = {"float32": "", "bfloat16": "-bf16", "float16": "-fp16"}


def backbone_dir_name(backbone: str, random_init: bool, backbone_dtype: str = "float32") -> str:
    """Output directory of a backbone.  A random-init or 16-bit run is tagged, so it never writes under the reference's own
    directory name."""
    return backbone + ("-randinit" if random_init else "") + _DTYPE_TAGS[backbone_dtype]


def _device() -> torch.device:
    return torch.device("cuda", torch.cuda.current_device())


def main(argv=None):
    parser = argparse.ArgumentParser("Calculating Matrix (B200-native path)")
    parser.add_argument("--path", default="data/mvtec_ad", type=str, help="Path to the dataset (unused for --dataset synthetic).")
    parser.add_argument("--backbone_names", nargs="+", default=["dino_vitbase8"], help="Architecture.")
    parser.add_argument("--layers_to_extract_from", nargs="+", default=["blocks.10", "blocks.11"])
    parser.add_argument("--pretrain_embed_dimension", default=2048, type=int)
    parser.add_argument("--target_embed_dimension", default=4096, type=int)
    parser.add_argument("--output_dir", default="outputs")
    parser.add_argument("--patchsize", type=int, default=3)
    parser.add_argument("--tau", type=float, nargs="+", default=[1.0], help="One or more taus (one distance pass serves all).")
    parser.add_argument("--train_ratio", type=float, default=1)
    parser.add_argument("--supervised", default="unsupervised", choices=["unsupervised", "supervised", "average"])
    parser.add_argument("--dataset", default="synthetic", type=str)
    parser.add_argument("--precision", default="auto")
    parser.add_argument("--synthetic_images", type=int, default=20)
    parser.add_argument("--synthetic_classes", type=int, default=4)
    parser.add_argument("--categories", nargs="+", default=["bottle"])
    parser.add_argument("--backbone_dtype", default="float32", choices=sorted(BACKBONE_DTYPES),
                        help="Run the backbone in this dtype; 16-bit feature maps go to the embed kernels as they are.")
    args = parser.parse_args(argv)
    print("\n".join("%s: %s" % (k, str(v)) for k, v in sorted(dict(vars(args)).items())))
    if args.dataset != "synthetic":
        raise SystemExit("only --dataset synthetic is available offline; for real data call "
                         "anomaly_clustering_b200.driver.make_category_data(..., test_dataloader=..., backbone=...)")
    device = _device()
    # --dataset synthetic is a shape / smoke run by construction: random-init network, said loudly, tagged output directory
    net = backbones.load(args.backbone_names[0], allow_random_init=True)
    backbone_dir = backbone_dir_name(args.backbone_names[0], getattr(net, "random_init", True), args.backbone_dtype)
    save_path = os.path.join(args.output_dir, args.dataset, backbone_dir, args.supervised)
    os.makedirs(save_path, exist_ok=True)
    rows = []
    for ci, category in enumerate(args.categories):
        loader, labels = synthetic_category(args.synthetic_images, args.synthetic_classes, seed=2023 + ci)
        train = None
        if args.supervised == "supervised":
            train, _ = synthetic_category(args.synthetic_images, 1, seed=4046 + ci)
        res = driver.make_category_data(args.path, category, args.pretrain_embed_dimension, args.target_embed_dimension,
                                        args.backbone_names, args.layers_to_extract_from, args.patchsize, save_path,
                                        train_ratio=args.train_ratio, tau=list(args.tau), supervised=args.supervised,
                                        dataset=args.dataset, test_dataloader=loader, train_dataloader=train, backbone=net,
                                        device=device, precision=args.precision,
                                        info_root=args.output_dir, allow_random_init=True,
                                        backbone_dtype=BACKBONE_DTYPES[args.backbone_dtype])
        from . import ops

        for (alpha, X), tau in zip(res, args.tau):
            Dm = ops.pairwise_l2(torch.from_numpy(X).to(device)).cpu().numpy()
            nmi, ari, f1, _, _ = cluster.calculate_metrics(Dm, labels)
            print("%s  tau=%g\nNMI: %s\nARI: %s\nF1:%s\n" % (category, tau, nmi, ari, f1))
            rows.append((category, tau, nmi, ari, f1))
    write_cli_csv(save_path, args.layers_to_extract_from, args.pretrain_embed_dimension, args.target_embed_dimension,
                  args.supervised, list(args.tau), rows)
    return rows


if __name__ == "__main__":
    main()
