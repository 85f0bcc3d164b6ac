"""AST-extraction of the reference's own pure-torch functions from a checkout of the original project (used by
tests/golden/make_golden.py to generate the golden vectors; the tests themselves read only tests/golden/).

Nothing is copied into the repo: the function source is read from the reference checkout, compiled in a scratch
namespace and called, so the vectors are produced by the reference's code itself."""
import ast
import os

import numpy as np
import torch

REF = None          # path of the reference checkout; set by the caller (make_golden.py --reference DIR)


def have_reference():
    return REF is not None and os.path.isdir(os.path.join(REF, 'src'))


def extract(relpath, names, extra_ns=None):
    src = open(os.path.join(REF, relpath)).read()
    tree = ast.parse(src)
    ns = {'torch': torch, 'np': np, 'F': torch.nn.functional}
    ns.update(extra_ns or {})
    for node in tree.body:
        if isinstance(node, (ast.FunctionDef, ast.ClassDef)) and node.name in names:
            code = compile(ast.Module(body=[node], type_ignores=[]), relpath, 'exec')
            exec(code, ns)
        elif isinstance(node, ast.Assign) and any(isinstance(t, ast.Name) and t.id in names for t in node.targets):
            code = compile(ast.Module(body=[node], type_ignores=[]), relpath, 'exec')
            exec(code, ns)
    return ns


def extract_method(relpath, cls_name, method, extra_ns=None):
    """one method of a class of the reference as a plain function (its `self` is whatever the caller passes)"""
    src = open(os.path.join(REF, relpath)).read()
    ns = {'torch': torch, 'np': np, 'F': torch.nn.functional}
    ns.update(extra_ns or {})
    for node in ast.parse(src).body:
        if isinstance(node, ast.ClassDef) and node.name == cls_name:
            for sub in node.body:
                if isinstance(sub, ast.FunctionDef) and sub.name == method:
                    sub.decorator_list = []
                    exec(compile(ast.Module(body=[sub], type_ignores=[]), relpath, 'exec'), ns)
                    return ns[method]
    raise KeyError(f'{cls_name}.{method} not found in {relpath}')
