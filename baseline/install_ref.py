"""Installs the UNMODIFIED reference (pytorch_bayesian 0.0.4, pure Python) into the git-ignored baseline/_ref/ so that it
travels to the GPU box with the repo snapshot (`/root/reference` does not exist there).

    python baseline/install_ref.py [--reference /root/reference]

1. `pip install --no-index --no-build-isolation --no-deps --target baseline/_ref <copy of the reference>` — the contract's
   recipe.  On this image it fails while generating metadata: setup.py lists `setup_requires=['pytest-runner']`, which no
   offline wheelhouse carries (the outcome is recorded in baseline/_ref/INSTALL.json).
2. Fallback, equivalent to what the install would have produced for a pure-Python distribution: the package directory
   `pytorch_bayesian/` copied file by file.  Nothing is edited.
Also copied, for the reference arm of bench.py: the three ELBO example model definitions
(examples/{MNIST,FashionMNIST,CIFAR10}/model.py).

Nothing under baseline/_ref is imported by the product package or the tests; users are bench.py --impl reference and
the "reference classes on CUDA" comparator.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
TARGET = os.path.join(HERE, "_ref")


def install(reference="/root/reference", quiet=False):
    if not os.path.isdir(os.path.join(reference, "pytorch_bayesian")):
        raise SystemExit(f"{reference} does not hold the reference checkout")
    if os.path.isdir(TARGET):
        shutil.rmtree(TARGET)
    os.makedirs(TARGET)
    record = {"reference": reference}
    with tempfile.TemporaryDirectory() as tmp:
        copy = os.path.join(tmp, "ref")
        shutil.copytree(reference, copy)            # /root/reference is read-only; setuptools writes egg-info
        cmd = [sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps",
               "--find-links", "/opt/wheelhouse", "--target", TARGET, copy]
        res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        record["pip_returncode"] = res.returncode
        record["pip_tail"] = res.stdout.strip().splitlines()[-6:]
    if not os.path.isdir(os.path.join(TARGET, "pytorch_bayesian")):
        record["method"] = "copy of the pure-Python package directory (pip could not build metadata offline)"
        shutil.copytree(os.path.join(reference, "pytorch_bayesian"), os.path.join(TARGET, "pytorch_bayesian"),
                        ignore=shutil.ignore_patterns("__pycache__"))
    else:
        record["method"] = "pip install --target"
    for name in ("MNIST", "FashionMNIST", "CIFAR10"):
        dst = os.path.join(TARGET, "examples", name)
        os.makedirs(dst, exist_ok=True)
        shutil.copy(os.path.join(reference, "examples", name, "model.py"), os.path.join(dst, "model.py"))
    with open(os.path.join(TARGET, "INSTALL.json"), "w") as fh:
        json.dump(record, fh, indent=1)
    if not quiet:
        print(json.dumps(record))
    return record


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", default="/root/reference")
    install(ap.parse_args().reference)
