"""Generate tests/golden/api_surface.json: the public Python surface of the reference (nrontsis/PILCO) that
tests/test_api_surface.py checks -- every module-level function, every class, and each class's methods with
their positional parameter names -- read from the reference's sources with ``ast`` (never imported).

    python tests/golden/make_api_surface.py <checkout of the reference>
"""
import ast
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
MODULES = {
    "pilco/models/mgpr.py": "pilco.models.mgpr",
    "pilco/models/smgpr.py": "pilco.models.smgpr",
    "pilco/models/pilco.py": "pilco.models.pilco",
    "pilco/controllers.py": "pilco.controllers",
    "pilco/rewards.py": "pilco.rewards",
    "safe_pilco_extension/rewards_safe.py": "safe_pilco_extension.rewards_safe",
    "safe_pilco_extension/safe_pilco.py": "safe_pilco_extension.safe_pilco",
}


def surface(path):
    tree = ast.parse(open(path).read())
    out = {"functions": [], "classes": {}}
    for node in tree.body:
        if isinstance(node, ast.FunctionDef):
            out["functions"].append(node.name)
        elif isinstance(node, ast.ClassDef):
            out["classes"][node.name] = [[item.name, [a.arg for a in item.args.args]]
                                         for item in node.body if isinstance(item, ast.FunctionDef)]
    return out


def main(ref):
    res = {modname: surface(os.path.join(ref, path)) for path, modname in MODULES.items()}
    with open(os.path.join(HERE, "api_surface.json"), "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main(sys.argv[1])
