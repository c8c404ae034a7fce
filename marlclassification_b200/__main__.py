"""Command line of the reference (``python -m marl_classification --run-id … train|test|infer``,
__main__.py:19-421) in front of the B200 episode: same modes, option names, defaults and
``marl.json`` / ``class_to_idx.json`` / ``models/nn_models_epoch_{e}.pt`` run-directory layout.
``--cuda`` is mandatory here (no CPU path).  Launch under ``torch.distributed.run`` to train data
parallel over the GPUs of one box."""
from __future__ import annotations

import argparse
import json
from os import makedirs
from os.path import abspath, dirname, exists, isdir, join
from typing import List, Optional, Sequence

from .registry import DATASET_REGISTRY

DEFAULT_ACTIONS = "[[1, 0], [-1, 0], [0, 1], [0, -1]]"


def parse_actions(text: str, dim: int) -> List[List[int]]:
    """``"[[1, 0], [-1, 0]]"`` -> ``[[1, 0], [-1, 0]]``; every move must be a list of ``dim``
    integers (__main__.py:329-345 validates the same with regular expressions)."""
    try:
        moves = json.loads(text)
    except json.JSONDecodeError as err:
        raise ValueError(f"Wrong action(s) : {text!r} ({err.msg})") from None
    well_formed = (isinstance(moves, list) and len(moves) > 0
                   and all(isinstance(m, list) and len(m) > 0 and all(type(v) is int for v in m) for m in moves))
    if not well_formed:
        raise ValueError(f"Wrong action(s) : {text!r} (expected a list of integer lists)")
    for i, m in enumerate(moves):
        assert len(m) == dim, f"Wrong space for action at index {i}"
    return moves


def build_parser() -> argparse.ArgumentParser:
    parser = argparse.ArgumentParser("Multi agent reinforcement learning for image classification - Main")
    parser.add_argument("--run-id", type=str, required=True, dest="run_id", help="name of this run (MLflow run name when MLflow is installed)")
    parser.add_argument("-a", "--agents", type=int, default=3, dest="agents", help="agents per image")
    parser.add_argument("--step", type=int, default=7, help="moves per episode (T)")
    parser.add_argument("--cuda", action="store_true", dest="cuda", help="Run on CUDA (required: this build has no CPU path)")
    modes = parser.add_subparsers(dest="main_choice", required=True)

    train = modes.add_parser("train")
    train.add_argument("--action", type=str, default=DEFAULT_ACTIONS, dest="action", help="move table as a JSON list of integer pairs")
    train.add_argument("--img-size", type=int, default=28, dest="img_size", help="side of the (square) images; recorded with the run")
    train.add_argument("--nb-class", type=int, default=10, dest="nb_class", help="number of classes")
    train.add_argument("-d", "--dim", type=int, default=2, help="dimension of an agent position (2 only)")
    train.add_argument("--f", type=int, default=7, help="side f of the observation window")
    train.add_argument("--ft-extr", type=str, choices=sorted(DATASET_REGISTRY), default="mnist", dest="ft_extr_str",
                       help="dataset / feature-extractor pair from the registry")
    for flag, dest, default, text in (
        ("--nb", "n_b", 64, "belief LSTM width n_b"),
        ("--na", "n_a", 16, "action LSTM width n_a"),
        ("--nm", "n_m", 16, "message width n_m"),
        ("--nmo", "n_m_o", 24, "decoded message width n_m_o"),
        ("--nd", "n_d", 4, "position feature width n_d"),
        ("--nlb", "n_l_b", 128, "hidden width of the prediction head"),
        ("--nla", "n_l_a", 128, "hidden width of the policy and critic heads"),
    ):
        train.add_argument(flag, type=int, default=default, dest=dest, help=text)
    train.add_argument("--res-folder", type=str, required=False,
                       default=abspath(join(dirname(abspath(__file__)), "..", "resources")),
                       help="directory holding downloaded/<dataset>")
    train.add_argument("-o", "--output-dir", type=str, required=True, dest="output_dir",
                       help="run directory (created): marl.json, class_to_idx.json, models/, pictures")
    train.add_argument("--batch-size", type=int, default=8, dest="batch_size",
                       help="images per optimisation step (the GLOBAL batch under torchrun)")
    train.add_argument("--lr", "--learning-rate", type=float, default=1e-3, dest="learning_rate", help="Adam step size")
    train.add_argument("--gamma", type=float, default=0.99, help="discount of the returns (0: the returns are the rewards, where the "
                       "original's closed form divides 0 by 0)")
    train.add_argument("--nb-epoch", type=int, default=10, dest="nb_epoch", help="passes over the training split")
    train.add_argument("--workers", type=int, default=6, help="DataLoader worker processes (train.py:95 uses 6)")
    train.add_argument("--resident", action="store_true",
                       help="decode the dataset once and keep it in HBM as bytes: no per-step host work or PCIe traffic")

    test = modes.add_parser("test")
    test.add_argument("--batch-size", type=int, default=8, dest="batch_size", help="images per forward episode")
    test.add_argument("--dataset-path", type=str, required=True, dest="dataset_path", help="image folder (one sub-directory per class)")
    test.add_argument("--img-size", type=int, default=28, dest="img_size", help="side of the (square) images; recorded with the run")
    test.add_argument("--json-path", type=str, required=True, dest="json_path", help="marl.json written by train")
    test.add_argument("--state-dict-path", type=str, required=True, dest="state_dict_path", help="models/nn_models_epoch_N.pt written by train")
    test.add_argument("-o", "--output-dir", type=str, required=True, dest="output_dir",
                      help="where the results go (created)")
    test.add_argument("--workers", type=int, default=8, help="DataLoader worker processes (eval.py:57 uses 8)")

    infer = modes.add_parser("infer")
    infer.add_argument("--images", type=str, nargs="+", required=True, dest="infer_images", help="image files or glob patterns")
    infer.add_argument("--json-path", type=str, required=True, dest="json_path", help="marl.json written by train")
    infer.add_argument("--state-dict-path", type=str, required=True, dest="state_dict_path", help="models/nn_models_epoch_N.pt written by train")
    infer.add_argument("--class2idx", type=str, required=True, dest="class_to_idx", help="class_to_idx.json written by train")
    infer.add_argument("-o", "--output-image-dir", type=str, required=True, dest="output_image_dir",
                       help="where the results go (created)")
    return parser


def _ensure_dir(path: str) -> None:
    if not exists(path):
        makedirs(path, exist_ok=True)
    if not isdir(path):
        raise NotADirectoryError(f'"{path}" is not a directory.')


def main(argv: Optional[Sequence[str]] = None) -> None:
    from .config import EvalConfig, InferConfig, MainConfig, ModelConfig, TrainConfig

    parser = build_parser()
    args = parser.parse_args(argv)
    main_config = MainConfig(step=args.step, run_id=args.run_id, cuda=args.cuda, nb_agent=args.agents)

    if args.main_choice == "train":
        try:
            actions = parse_actions(args.action, args.dim)
        except ValueError as err:
            parser.error(str(err))
        model_config = ModelConfig(
            ft_extr_str=args.ft_extr_str, window_size=args.f, hidden_size_belief=args.n_b, hidden_size_action=args.n_a,
            hidden_size_msg=args.n_m, hidden_size_msg_output=args.n_m_o, hidden_size_state=args.n_d, state_dim=args.dim,
            actions=actions, nb_class=args.nb_class, hidden_size_linear_belief=args.n_l_b,
            hidden_size_linear_action=args.n_l_a,
        )
        train_config = TrainConfig(
            img_size=args.img_size, nb_epoch=args.nb_epoch, learning_rate=args.learning_rate, batch_size=args.batch_size,
            resources_dir=args.res_folder, output_dir=args.output_dir, gamma=args.gamma,
        )
        _ensure_dir(args.output_dir)
        from .train import train_main

        train_main(main_config, model_config, train_config, num_workers=args.workers, resident=args.resident)
    elif args.main_choice == "test":
        eval_config = EvalConfig(
            img_size=args.img_size, state_dict_path=args.state_dict_path, batch_size=args.batch_size,
            json_path=args.json_path, dataset_path=args.dataset_path, output_dir=args.output_dir,
        )
        _ensure_dir(args.output_dir)
        from .eval import eval_main

        eval_main(main_config, eval_config, num_workers=args.workers)
    else:
        infer_config = InferConfig(
            state_dict_path=args.state_dict_path, json_path=args.json_path, images_path=args.infer_images,
            output_dir=args.output_image_dir, class_to_idx=args.class_to_idx,
        )
        _ensure_dir(args.output_image_dir)
        from .infer import infer_main

        infer_main(main_config, infer_config)


if __name__ == "__main__":
    main()
