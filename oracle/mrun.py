"""mrun -- a small interpreter for the MATLAB subset used by the reference's oracle files.

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.

The reference's tests compare the Python code with ``tests/Matlab Code/*.m`` executed live in Octave
(oct2py).  Without Octave, this module executes those ``.m`` files -- by default the unmodified copies
under ``tests/reference_tests/Matlab Code`` (checksums in ``tests/reference_tests/sha256sums.txt``): it is
the "reference itself run here" that pins ``oracle/matlab_port.py`` and generates ``tests/golden/*.npz``
(``tests/golden/make_golden.py``).

Supported: function files with multiple outputs, nargin/nargout, if/elseif/else, for, return, persistent
(ignored), struct field access/assignment, N-d indexing with ``end`` and ``:``, indexed assignment with
auto-growth, matrix literals with MATLAB's whitespace rules, ranges, the operators
``+ - * / \\ .* ./ .^ ^ ' == ~= < <= > >= && || & | ~`` and the builtins listed in ``BUILTINS``.
Statements are parsed lazily (only when executed), so unexecuted derivative blocks need not be supported.
"""
import os
import re

import numpy as np

MDIR_DEFAULT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "reference_tests", "Matlab Code")


class MError(Exception):
    pass


# --------------------------------------------------------------------------------------------------
# tokenizer
# --------------------------------------------------------------------------------------------------
TOK_RE = re.compile(r"""
    (?P<num>(\d+\.?\d*|\.\d+)([eE][+-]?\d+)?) |
    (?P<id>[A-Za-z_]\w*) |
    (?P<op>\.\*|\./|\.\\|\.\^|\.'|==|~=|<=|>=|&&|\|\||[-+*/\\^'<>=~&|:;,()\[\]{}.@])
""", re.X)


class Tok:
    __slots__ = ("kind", "val", "ws_before", "ws_after")

    def __init__(self, kind, val, ws_before):
        self.kind, self.val, self.ws_before, self.ws_after = kind, val, ws_before, False

    def __repr__(self):
        return "%s:%r" % (self.kind, self.val)


def tokenize(src):
    toks, i, n = [], 0, len(src)
    while i < n:
        c = src[i]
        ws = False
        while i < n and src[i] in " \t":
            i += 1
            ws = True
        if i >= n:
            break
        c = src[i]
        if toks:
            toks[-1].ws_after = ws
        if c == "'":
            prev = toks[-1] if toks else None
            is_transpose = prev is not None and not ws and (prev.kind in ("num", "id") or prev.val in (")", "]", "'", ".'", "}"))
            if prev is not None and ws and (prev.kind in ("num", "id") or prev.val in (")", "]", "'")):
                is_transpose = False
            if not is_transpose:
                j = i + 1
                buf = []
                while j < n:
                    if src[j] == "'":
                        if j + 1 < n and src[j + 1] == "'":
                            buf.append("'"); j += 2; continue
                        break
                    buf.append(src[j]); j += 1
                toks.append(Tok("str", "".join(buf), ws))
                i = j + 1
                continue
        m = TOK_RE.match(src, i)
        if not m:
            raise MError("cannot tokenize at %r" % src[i:i + 20])
        kind = m.lastgroup
        if kind == "num":
            toks.append(Tok("num", float(m.group("num")), ws))
        elif kind == "id":
            toks.append(Tok("id", m.group("id"), ws))
        else:
            toks.append(Tok("op", m.group("op"), ws))
        i = m.end()
    return toks


# --------------------------------------------------------------------------------------------------
# values
# --------------------------------------------------------------------------------------------------
def A(x):
    """to MATLAB value: ndarray with ndim >= 2"""
    if isinstance(x, (dict, str)) or callable(x):
        return x
    a = np.asarray(x, dtype=np.float64)
    if a.ndim == 0:
        return a.reshape(1, 1)
    if a.ndim == 1:
        return a.reshape(1, -1)
    return a


def scalar(v):
    a = np.asarray(v)
    if a.size != 1:
        raise MError("expected scalar, got shape %s" % (a.shape,))
    return float(a.reshape(-1)[0])


def truth(v):
    a = np.asarray(v)
    return a.size > 0 and bool(np.all(a != 0))


class Colon:
    pass


COLON = Colon()


class EndMarker:
    pass


# --------------------------------------------------------------------------------------------------
# expression parser / evaluator (evaluates while parsing)
# --------------------------------------------------------------------------------------------------
class Expr:
    def __init__(self, toks, interp, scope):
        self.t, self.i, self.I, self.scope = toks, 0, interp, scope
        self.end_stack = []          # (array, dim_index, n_indices) for `end`
        self.in_matrix = 0
        self.paren_depth_in_matrix = []

    def peek(self):
        return self.t[self.i] if self.i < len(self.t) else None

    def next(self):
        tk = self.peek()
        self.i += 1
        return tk

    def accept(self, val):
        tk = self.peek()
        if tk is not None and tk.kind == "op" and tk.val == val:
            self.i += 1
            return True
        return False

    def expect(self, val):
        if not self.accept(val):
            raise MError("expected %r at token %d of %r" % (val, self.i, self.t))

    # precedence climbing -------------------------------------------------------------------------
    def parse(self):
        return self.p_oror()

    def p_oror(self):
        v = self.p_andand()
        while self.accept("||"):
            r = self.p_andand()
            v = A(float(truth(v) or truth(r)))
        return v

    def p_andand(self):
        v = self.p_or()
        while self.accept("&&"):
            r = self.p_or()
            v = A(float(truth(v) and truth(r)))
        return v

    def p_or(self):
        v = self.p_and()
        while self.peek() is not None and self.peek().kind == "op" and self.peek().val == "|":
            self.next()
            r = self.p_and()
            v = A(np.logical_or(v != 0, r != 0).astype(float))
        return v

    def p_and(self):
        v = self.p_cmp()
        while self.peek() is not None and self.peek().kind == "op" and self.peek().val == "&":
            self.next()
            r = self.p_cmp()
            v = A(np.logical_and(v != 0, r != 0).astype(float))
        return v

    def p_cmp(self):
        v = self.p_range()
        while True:
            tk = self.peek()
            if tk is None or tk.kind != "op" or tk.val not in ("==", "~=", "<", "<=", ">", ">="):
                return v
            self.next()
            r = self.p_range()
            f = {"==": np.equal, "~=": np.not_equal, "<": np.less, "<=": np.less_equal,
                 ">": np.greater, ">=": np.greater_equal}[tk.val]
            v = A(f(v, r).astype(float))

    def _elem_break(self):
        """inside a matrix literal: does the upcoming token start a new element?"""
        if not self.in_matrix or self.paren_depth_in_matrix[-1] != 0:
            return False
        tk = self.peek()
        if tk is None:
            return False
        if tk.kind == "op" and tk.val in ("+", "-") and tk.ws_before and not tk.ws_after:
            return True
        return False

    def p_range(self):
        v = self.p_add()
        tk = self.peek()
        if tk is not None and tk.kind == "op" and tk.val == ":" and not self._colon_is_index():
            self.next()
            b = self.p_add()
            if self.peek() is not None and self.peek().kind == "op" and self.peek().val == ":":
                self.next()
                c = self.p_add()
                return A(np.arange(scalar(v), scalar(c) + 0.5 * np.sign(scalar(b)) * 1e-9 + (1e-12 if scalar(b) > 0 else -1e-12), scalar(b)))
            lo, hi = scalar(v), scalar(b)
            return A(np.arange(lo, hi + 1e-9, 1.0)) if hi >= lo else np.zeros((1, 0))
        return v

    def _colon_is_index(self):
        return False

    def p_add(self):
        v = self.p_mul()
        while True:
            tk = self.peek()
            if tk is None or tk.kind != "op" or tk.val not in ("+", "-"):
                return v
            if self._elem_break():
                return v
            self.next()
            r = self.p_mul()
            v = A(v + r) if tk.val == "+" else A(v - r)

    def p_mul(self):
        v = self.p_unary()
        while True:
            tk = self.peek()
            if tk is None or tk.kind != "op" or tk.val not in ("*", "/", "\\", ".*", "./", ".\\"):
                return v
            self.next()
            r = self.p_unary()
            v = A(self.mul_op(tk.val, v, r))

    @staticmethod
    def mul_op(op, a, b):
        if op == ".*":
            return a * b
        if op == "./":
            return a / b
        if op == ".\\":
            return b / a
        if op == "*":
            if a.size == 1 or b.size == 1:
                return a * b
            return a @ b
        if op == "/":
            if b.size == 1:
                return a / b
            return np.linalg.solve(b.T, a.T).T          # a / b = a * inv(b)
        if op == "\\":
            if a.size == 1:
                return b / a
            return np.linalg.solve(a, b)
        raise MError(op)

    def p_unary(self):
        tk = self.peek()
        if tk is not None and tk.kind == "op" and tk.val in ("-", "+", "~"):
            self.next()
            v = self.p_unary()
            if tk.val == "-":
                return A(-v)
            if tk.val == "~":
                return A((np.asarray(v) == 0).astype(float))
            return v
        return self.p_power()

    def p_power(self):
        v = self.p_postfix()
        while True:
            tk = self.peek()
            if tk is None or tk.kind != "op" or tk.val not in ("^", ".^"):
                return v
            self.next()
            # exponent: unary minus allowed
            neg = False
            if self.peek() is not None and self.peek().kind == "op" and self.peek().val in ("-", "+"):
                neg = self.next().val == "-"
            r = self.p_postfix()
            if neg:
                r = A(-r)
            if tk.val == ".^" or (v.size == 1 and r.size == 1):
                v = A(np.power(v, r))
            else:
                v = A(np.linalg.matrix_power(v, int(scalar(r))))

    def p_postfix(self):
        v = self.p_primary()
        while True:
            tk = self.peek()
            if tk is None or tk.kind != "op":
                return v
            if tk.val in ("'", ".'"):
                self.next()
                if isinstance(v, np.ndarray):
                    if v.ndim != 2:
                        raise MError("transpose of N-d array")
                    v = v.T
                continue
            return v

    def parse_args(self, target):
        """parse `( ... )` argument list; target is the array being indexed (for `end`) or None"""
        self.expect("(")
        if self.in_matrix:
            self.paren_depth_in_matrix[-1] += 1
        args = []
        # count the number of indices by a look-ahead scan (needed for `end` in the last position)
        depth, nidx, j = 0, 1, self.i
        while j < len(self.t):
            tk = self.t[j]
            if tk.kind == "op":
                if tk.val in ("(", "[", "{"):
                    depth += 1
                elif tk.val in (")", "]", "}"):
                    if depth == 0:
                        break
                    depth -= 1
                elif tk.val == "," and depth == 0:
                    nidx += 1
            j += 1
        if self.accept(")"):
            if self.in_matrix:
                self.paren_depth_in_matrix[-1] -= 1
            return args
        k = 0
        while True:
            tk = self.peek()
            nxt = self.t[self.i + 1] if self.i + 1 < len(self.t) else None
            if tk is not None and tk.kind == "op" and tk.val == ":" and nxt is not None and nxt.kind == "op" and nxt.val in (",", ")"):
                self.next()
                args.append(COLON)
            else:
                self.end_stack.append((target, k, nidx))
                saved = self.in_matrix
                self.in_matrix = 0                       # whitespace rules do not apply inside parentheses
                args.append(self.parse())
                self.in_matrix = saved
                self.end_stack.pop()
            k += 1
            if self.accept(","):
                continue
            self.expect(")")
            break
        if self.in_matrix:
            self.paren_depth_in_matrix[-1] -= 1
        return args

    def p_primary(self):
        tk = self.next()
        if tk is None:
            raise MError("unexpected end of expression")
        if tk.kind == "num":
            return A(tk.val)
        if tk.kind == "str":
            return tk.val
        if tk.kind == "op":
            if tk.val == "(":
                saved = self.in_matrix
                self.in_matrix = 0
                v = self.parse()
                self.in_matrix = saved
                self.expect(")")
                return v
            if tk.val == "[":
                return self.p_matrix()
            if tk.val == "@":
                name = self.next().val
                return self.I.function_handle(name)
            if tk.val == ":":
                return COLON
            raise MError("unexpected %r" % tk.val)
        name = tk.val
        if name == "end" and self.end_stack:
            arr, k, nidx = self.end_stack[-1]
            if arr is None:
                raise MError("`end` outside indexing")
            return A(float(dim_for_end(arr, k, nidx)))
        if name == "true":
            return A(1.0)
        if name == "false":
            return A(0.0)
        if name in self.scope:
            v = self.scope[name]
            return self.p_chain(v)
        if name == "nargin":
            return A(float(self.scope["__nargin__"]))
        if name == "nargout":
            return A(float(self.scope["__nargout__"]))
        # function call
        args = []
        nxt = self.peek()
        if nxt is not None and nxt.kind == "op" and nxt.val == "(" and not (self.in_matrix and nxt.ws_before and self.paren_depth_in_matrix[-1] == 0):
            args = self.parse_args(None)
        out = self.I.call(name, args, 1)
        return self.p_chain(out[0] if isinstance(out, tuple) else out)

    def p_chain(self, v):
        """field access / indexing chain on a value"""
        while True:
            tk = self.peek()
            if tk is None or tk.kind != "op":
                return v
            if tk.val == "." and isinstance(v, dict):
                self.next()
                v = v[self.next().val]
                continue
            if tk.val == "(" and not (self.in_matrix and tk.ws_before and self.paren_depth_in_matrix[-1] == 0):
                if not isinstance(v, np.ndarray):
                    raise MError("indexing into non-array")
                args = self.parse_args(v)
                v = index_get(v, args)
                continue
            return v

    def p_matrix(self):
        self.in_matrix += 1
        self.paren_depth_in_matrix.append(0)
        rows, cur = [], []
        while True:
            tk = self.peek()
            if tk is None:
                raise MError("unterminated [")
            if tk.kind == "op" and tk.val == "]":
                self.next()
                break
            if tk.kind == "op" and tk.val == ";":
                self.next()
                rows.append(cur); cur = []
                continue
            if tk.kind == "op" and tk.val == ",":
                self.next()
                continue
            cur.append(self.parse())
        rows.append(cur)
        self.in_matrix -= 1
        self.paren_depth_in_matrix.pop()
        rows = [r for r in rows if r]
        if not rows:
            return np.zeros((0, 0))
        hrows = []
        for r in rows:
            parts = [p for p in r if not (isinstance(p, np.ndarray) and p.size == 0)]
            if not parts:
                continue
            hrows.append(np.concatenate([A(p) for p in parts], axis=1))
        if not hrows:
            return np.zeros((0, 0))
        return np.concatenate(hrows, axis=0)


def dim_for_end(arr, k, nidx):
    shp = arr.shape
    if nidx == 1:
        return arr.size
    if k < nidx - 1:
        return shp[k] if k < len(shp) else 1
    return int(np.prod(shp[k:])) if k < len(shp) else 1


def _idx(v, n):
    if isinstance(v, Colon):
        return np.arange(n)
    a = np.asarray(v, dtype=np.float64).reshape(-1)
    return (np.round(a) - 1).astype(int)


def index_get(arr, args):
    if len(args) == 0:
        return arr
    if len(args) == 1:
        a = args[0]
        flat = arr.reshape(-1, order="F")
        if isinstance(a, Colon):
            return flat.reshape(-1, 1)
        ia = np.asarray(a)
        res = flat[_idx(a, arr.size)]
        if arr.ndim == 2 and (arr.shape[0] == 1 or arr.shape[1] == 1) and (ia.ndim < 2 or min(ia.shape) == 1):
            return res.reshape(1, -1) if arr.shape[0] == 1 and arr.shape[1] != 1 else (res.reshape(-1, 1) if arr.shape[1] == 1 and arr.shape[0] != 1 else A(res).reshape(ia.shape if ia.ndim == 2 else (1, -1)))
        return res.reshape(ia.shape if ia.ndim >= 2 else (1, -1), order="F")
    shp = list(arr.shape) + [1] * (len(args) - arr.ndim)
    if len(args) < arr.ndim:
        shp = list(arr.shape[:len(args) - 1]) + [int(np.prod(arr.shape[len(args) - 1:]))]
    a2 = arr.reshape(shp, order="F")
    idx = [_idx(a, shp[k]) for k, a in enumerate(args)]
    out = a2[np.ix_(*idx)]
    while out.ndim > 2 and out.shape[-1] == 1:
        out = out.reshape(out.shape[:-1], order="F")
    return out


def index_set(arr, args, val):
    val = A(val) if not isinstance(val, np.ndarray) else val
    if arr is None:
        arr = np.zeros((0, 0))
    if len(args) == 1:
        a = args[0]
        if isinstance(a, Colon):
            arr = arr.copy()
            arr.reshape(-1, order="F")[:] = np.asarray(val).reshape(-1, order="F")
            return arr
        ii = _idx(a, arr.size)
        need = int(ii.max()) + 1 if ii.size else 0
        if need > arr.size:
            if arr.size == 0:
                arr = np.zeros((1, need))
            elif arr.shape[0] == 1:
                arr = np.concatenate([arr, np.zeros((1, need - arr.shape[1]))], axis=1)
            elif arr.shape[1] == 1:
                arr = np.concatenate([arr, np.zeros((need - arr.shape[0], 1))], axis=0)
            else:
                raise MError("cannot grow matrix with linear index")
        flat = arr.reshape(-1, order="F").copy()
        v = np.asarray(val, dtype=np.float64).reshape(-1, order="F")
        flat[ii] = v if v.size != 1 else v[0]
        return flat.reshape(arr.shape, order="F")
    nd = max(len(args), arr.ndim)
    shp = list(arr.shape) + [1] * (nd - arr.ndim)
    vshape = list(np.asarray(val).shape)
    idx, newshp = [], list(shp)
    vdim = 0
    for k, a in enumerate(args):
        if isinstance(a, Colon):
            n = shp[k]
            if n == 0 or (arr.size == 0):
                # take from value
                nonsingle = [d for d in vshape]
                n = vshape[vdim] if vdim < len(vshape) else 1
            idx.append(np.arange(n))
        else:
            idx.append(_idx(a, shp[k]))
        if idx[-1].size:
            newshp[k] = max(newshp[k], int(idx[-1].max()) + 1)
        vdim += 1
    if newshp != shp or arr.size == 0:
        big = np.zeros(newshp)
        if arr.size:
            big[tuple(slice(0, s) for s in shp)] = arr.reshape(shp, order="F")
        arr2 = big
    else:
        arr2 = arr.reshape(shp, order="F").copy()
    v = np.asarray(val, dtype=np.float64)
    tgt_shape = [len(i) for i in idx]
    if v.size == 1:
        arr2[np.ix_(*idx)] = v.reshape(-1)[0]
    else:
        vs = [d for d in v.shape if d != 1]
        ts = [d for d in tgt_shape if d != 1]
        if vs != ts:
            raise MError("assignment dimension mismatch %s vs %s" % (v.shape, tgt_shape))
        arr2[np.ix_(*idx)] = v.reshape(tgt_shape, order="F") if v.ndim <= 2 and len(tgt_shape) > 2 else _reshape_like(v, tgt_shape)
    while arr2.ndim > 2 and arr2.shape[-1] == 1:
        arr2 = arr2.reshape(arr2.shape[:-1])
    return arr2


def _reshape_like(v, tgt_shape):
    # map the non-singleton dims of v onto the non-singleton dims of the target, preserving order
    return v.reshape([d for d in tgt_shape], order="F") if v.ndim != len(tgt_shape) or list(v.shape) != list(tgt_shape) else v


# --------------------------------------------------------------------------------------------------
# builtins
# --------------------------------------------------------------------------------------------------
def _dims(args):
    if len(args) == 1:
        a = np.asarray(args[0]).reshape(-1)
        return (int(a[0]), int(a[0])) if a.size == 1 else tuple(int(x) for x in a)
    return tuple(int(scalar(a)) for a in args)


def b_size(args, nout):
    a = args[0]
    shp = list(a.shape) if isinstance(a, np.ndarray) else [1, 1]
    if len(args) == 2:
        k = int(scalar(args[1])) - 1
        return A(float(shp[k] if k < len(shp) else 1))
    if nout <= 1:
        return A(np.array(shp, dtype=float))
    out = []
    for k in range(nout):
        if k < nout - 1:
            out.append(A(float(shp[k] if k < len(shp) else 1)))
        else:
            out.append(A(float(np.prod(shp[k:])) if k < len(shp) else 1.0))
    return tuple(out)


def b_sum(args, nout):
    a = args[0]
    if len(args) == 2:
        ax = int(scalar(args[1])) - 1
    else:
        ax = 0 if a.shape[0] != 1 else 1
    return A(a.sum(axis=ax, keepdims=True)) if a.ndim == 2 else A(a.sum(axis=ax))


def b_diag(args, nout):
    a = args[0]
    if a.shape[0] == 1 or a.shape[1] == 1:
        return np.diag(a.reshape(-1))
    return np.diag(a).reshape(-1, 1)


def b_chol(args, nout):
    return np.linalg.cholesky(args[0]).T                 # upper triangular R with R'R = A


def b_minmax(f):
    def g(args, nout):
        if len(args) == 2:
            return A(f(args[0], args[1]))
        a = args[0]
        return A(f.reduce(a.reshape(-1))) if min(a.shape) == 1 else A(f.reduce(a, axis=0))
    return g


def b_bsxfun(args, nout):
    return A(args[0](args[1], args[2]))


def b_isfield(args, nout):
    return A(float(isinstance(args[0], dict) and args[1] in args[0]))


def b_any(args, nout):
    a = np.asarray(args[0])
    return A(float(np.any(a != 0))) if min(a.shape) == 1 else A(np.any(a != 0, axis=0).astype(float))


BUILTINS = {
    "size": b_size, "sum": b_sum, "diag": b_diag, "chol": b_chol, "bsxfun": b_bsxfun, "isfield": b_isfield,
    "zeros": lambda a, n: np.zeros(_dims(a)), "ones": lambda a, n: np.ones(_dims(a)),
    "eye": lambda a, n: np.eye(*_dims(a)),
    "exp": lambda a, n: A(np.exp(a[0])), "log": lambda a, n: A(np.log(a[0])), "sqrt": lambda a, n: A(np.sqrt(a[0])),
    "sin": lambda a, n: A(np.sin(a[0])), "cos": lambda a, n: A(np.cos(a[0])), "abs": lambda a, n: A(np.abs(a[0])),
    "det": lambda a, n: A(np.linalg.det(a[0])), "inv": lambda a, n: np.linalg.inv(a[0]),
    "numel": lambda a, n: A(float(np.asarray(a[0]).size)), "length": lambda a, n: A(float(max(np.asarray(a[0]).shape) if np.asarray(a[0]).size else 0)),
    "isempty": lambda a, n: A(float(np.asarray(a[0]).size == 0)),
    "min": b_minmax(np.minimum), "max": b_minmax(np.maximum), "any": b_any,
    "linspace": lambda a, n: A(np.linspace(scalar(a[0]), scalar(a[1]), int(scalar(a[2])))),
    "kron": lambda a, n: np.kron(a[0], a[1]),
    "reshape": lambda a, n: np.asarray(a[0]).reshape(_dims(a[1:]), order="F"),
    "trace": lambda a, n: A(np.trace(a[0])),
}
HANDLES = {"plus": np.add, "minus": np.subtract, "times": np.multiply, "rdivide": np.divide}


# --------------------------------------------------------------------------------------------------
# statements / interpreter
# --------------------------------------------------------------------------------------------------
class Return(Exception):
    pass


class MFunction:
    def __init__(self, name, outs, ins, body):
        self.name, self.outs, self.ins, self.body = name, outs, ins, body


def strip_comment(line):
    out, in_str, i = [], False, 0
    while i < len(line):
        c = line[i]
        if c == "'" :
            prev = line[i - 1] if i else " "
            if in_str:
                in_str = False
            elif not (prev.isalnum() or prev in ")]}'._"):
                in_str = True
        if c == "%" and not in_str:
            break
        out.append(c)
        i += 1
    return "".join(out).rstrip()


def split_statements(text):
    """-> list of statement strings (continuations joined, ';'/',' separated statements split at depth 0)"""
    lines, buf = [], ""
    for raw in text.splitlines():
        ln = strip_comment(raw)
        if ln.rstrip().endswith("..."):
            buf += ln.rstrip()[:-3] + " "
            continue
        buf += ln
        if buf.strip():
            lines.append(buf.strip())
        buf = ""
    stmts = []
    for ln in lines:
        depth, cur, in_str, k = 0, "", False, 0
        first = re.match(r"[A-Za-z_]\w*", ln)
        while k < len(ln):
            c = ln[k]
            if c == "'":
                prev = ln[k - 1] if k else " "
                if in_str:
                    in_str = False
                elif not (prev.isalnum() or prev in ")]}'._"):
                    in_str = True
            if not in_str:
                if c in "([{":
                    depth += 1
                elif c in ")]}":
                    depth -= 1
                elif c == ";" and depth == 0:
                    if cur.strip():
                        stmts.append(cur.strip() + ";")
                    cur = ""; k += 1
                    continue
                elif c == "," and depth == 0 and re.match(r"\s*(if|for|end|else|elseif|return)\b", cur.strip() + " x") is None and False:
                    pass
            cur += c
            k += 1
        if cur.strip():
            stmts.append(cur.strip())
    # split "if cond, stmt; end" one-liners and "end" trailing keywords
    out = []
    for s in stmts:
        cut = _top_level_comma(s) if re.match(r"^if\b", s) else -1
        if cut > 0:
            out.append(s[:cut].strip())
            for part in re.split(r";\s*", s[cut + 1:]):
                part = part.strip()
                if part:
                    out.extend(_split_kw(part))
            continue
        out.extend(_split_kw(s))
    return out


def _top_level_comma(s):
    depth = 0
    for k, c in enumerate(s):
        if c in "([{":
            depth += 1
        elif c in ")]}":
            depth -= 1
        elif c == "," and depth == 0:
            return k
    return -1


def _balanced(s):
    return s.count("(") == s.count(")") and s.count("[") == s.count("]")


def _split_kw(s):
    """'x = 1; else y = 2; end' pieces after ';' splitting -> separate keyword statements"""
    res = []
    s = s.strip()
    m = re.match(r"^(else|end|return)\b\s*;?\s*(.*)$", s)
    while m and m.group(2):
        res.append(m.group(1))
        s = m.group(2).strip()
        m = re.match(r"^(else|end|return)\b\s*;?\s*(.*)$", s)
    m2 = re.match(r"^(.*\S)\s+end;?$", s)
    if m2 and not re.match(r"^(if|for|while|function)\b", s) and _balanced(m2.group(1)) and "(" not in m2.group(1).split("=")[-1][-1:]:
        # statement followed by trailing `end` on the same line (e.g. "[M,S,V] = gp0(...); return; end")
        res.append(m2.group(1)); res.append("end")
        return res
    if s:
        res.append(s)
    return res


class Interp:
    def __init__(self, mdir=MDIR_DEFAULT):
        self.mdir, self.funcs = mdir, {}

    def function_handle(self, name):
        if name in HANDLES:
            return HANDLES[name]
        return lambda *a: self.call(name, list(a), 1)

    def load(self, name):
        if name in self.funcs:
            return self.funcs[name]
        path = os.path.join(self.mdir, name + ".m")
        if not os.path.exists(path):
            raise MError("unknown function %s" % name)
        stmts = split_statements(open(path).read())
        hdr = None
        for k, s in enumerate(stmts):
            if s.startswith("function"):
                hdr = k
                break
        if hdr is None:
            raise MError("no function header in %s" % path)
        h = stmts[hdr].rstrip(";")
        m = re.match(r"function\s+(?:\[(.*?)\]|(\w+))\s*=\s*(\w+)\s*\((.*?)\)", h)
        outs = [o for o in re.split(r"[,\s]+", (m.group(1) or m.group(2)).strip()) if o]
        ins = [a.strip() for a in m.group(4).split(",") if a.strip()]
        fn = MFunction(m.group(3), outs, ins, stmts[hdr + 1:])
        self.funcs[name] = fn
        return fn

    def call(self, name, args, nout):
        if name in BUILTINS:
            return BUILTINS[name](args, nout)
        fn = self.load(name)
        scope = {"__nargin__": len(args), "__nargout__": nout}
        for k, a in enumerate(args):
            scope[fn.ins[k]] = a
        try:
            self.exec_block(fn.body, 0, len(fn.body), scope)
        except Return:
            pass
        outs = tuple(scope[o] for o in fn.outs[:max(nout, 1)])
        return outs

    # ---- block structure by keywords only (lazy expression parsing) ------------------------------
    @staticmethod
    def kw(s):
        m = re.match(r"^(if|elseif|else|for|while|end|function|return|persistent|break)\b", s)
        return m.group(1) if m else None

    def find_block(self, body, i):
        """i at an if/for: returns index of the matching end and the positions of elseif/else at depth 0"""
        depth, marks, j = 0, [], i + 1
        while j < len(body):
            k = self.kw(body[j])
            if k in ("if", "for", "while"):
                depth += 1
            elif k == "end":
                if depth == 0:
                    return j, marks
                depth -= 1
            elif k in ("elseif", "else") and depth == 0:
                marks.append(j)
            j += 1
        raise MError("unterminated block starting at %r" % body[i])

    def exec_block(self, body, lo, hi, scope):
        i = lo
        while i < hi:
            s = body[i]
            k = self.kw(s)
            if k == "function":
                return                                   # start of a sub-function / commented helper
            if k == "persistent" or s.rstrip(";") == "":
                i += 1
                continue
            if k == "return":
                raise Return()
            if k == "if":
                end, marks = self.find_block(body, i)
                bounds = [i] + marks + [end]
                done = False
                for b in range(len(bounds) - 1):
                    head = body[bounds[b]]
                    hk = self.kw(head)
                    if hk == "else":
                        cond = True
                    else:
                        cond = truth(self.eval(re.sub(r"^(if|elseif)\b", "", head).rstrip(";,").strip(), scope))
                    if cond:
                        self.exec_block(body, bounds[b] + 1, bounds[b + 1], scope)
                        done = True
                        break
                i = end + 1
                continue
            if k == "for":
                end, _ = self.find_block(body, i)
                m = re.match(r"^for\s+(\w+)\s*=\s*(.*)$", s.rstrip(";"))
                rng = self.eval(m.group(2), scope)
                for col in range(rng.shape[1]):
                    scope[m.group(1)] = A(rng[:, col]) if rng.shape[0] > 1 else A(rng[0, col])
                    self.exec_block(body, i + 1, end, scope)
                i = end + 1
                continue
            if k == "end":
                i += 1
                continue
            self.exec_statement(s, scope)
            i += 1

    def eval(self, src, scope):
        ex = Expr(tokenize(src), self, scope)
        v = ex.parse()
        if ex.i != len(ex.t):
            raise MError("trailing tokens in %r at %d: %s" % (src, ex.i, ex.t[ex.i:]))
        return v

    # ---- assignment --------------------------------------------------------------------------------
    def exec_statement(self, s, scope):
        s = s.rstrip(";").strip()
        toks = tokenize(s)
        # find top-level '='
        depth, eq = 0, None
        for k, tk in enumerate(toks):
            if tk.kind == "op":
                if tk.val in ("(", "[", "{"):
                    depth += 1
                elif tk.val in (")", "]", "}"):
                    depth -= 1
                elif tk.val == "=" and depth == 0:
                    eq = k
                    break
        if eq is None:
            self.eval(s, scope)
            return
        lhs, rhs = toks[:eq], toks[eq + 1:]
        if lhs and lhs[0].kind == "op" and lhs[0].val == "[":
            targets = self.split_targets(lhs[1:-1])
            # rhs must be a single function call
            name = rhs[0].val
            ex = Expr(rhs, self, scope)
            ex.i = 1
            args = ex.parse_args(None) if ex.peek() is not None else []
            outs = self.call(name, args, len(targets))
            if not isinstance(outs, tuple):
                outs = (outs,)
            for tgt, val in zip(targets, outs):
                self.assign(tgt, val, scope)
            return
        ex = Expr(rhs, self, scope)
        val = ex.parse()
        if ex.i != len(rhs):
            raise MError("trailing tokens in %r" % s)
        self.assign(lhs, val, scope)

    @staticmethod
    def split_targets(toks):
        out, cur, depth = [], [], 0
        for tk in toks:
            if tk.kind == "op" and tk.val in ("(", "["):
                depth += 1
            elif tk.kind == "op" and tk.val in (")", "]"):
                depth -= 1
            if depth == 0 and ((tk.kind == "op" and tk.val == ",") or (cur and tk.ws_before and not (tk.kind == "op" and tk.val in (")", "]", ".", "(")) and not (cur[-1].kind == "op" and cur[-1].val == "."))):
                if tk.kind == "op" and tk.val == ",":
                    if cur:
                        out.append(cur)
                    cur = []
                    continue
                out.append(cur)
                cur = [tk]
                continue
            cur.append(tk)
        if cur:
            out.append(cur)
        return out

    def assign(self, lhs, val, scope):
        name = lhs[0].val
        if len(lhs) == 1:
            scope[name] = val
            return
        if lhs[1].kind == "op" and lhs[1].val == ".":
            # struct field path: a.b.c = val   (optionally with trailing index on the last field)
            path, k = [name], 1
            while k < len(lhs) and lhs[k].kind == "op" and lhs[k].val == ".":
                path.append(lhs[k + 1].val)
                k += 2
            obj = scope.setdefault(path[0], {})
            for f in path[1:-1]:
                obj = obj.setdefault(f, {})
            if k < len(lhs):
                ex = Expr(lhs[k:], self, scope)
                args = ex.parse_args(obj.get(path[-1]))
                obj[path[-1]] = index_set(obj.get(path[-1]), args, val)
            else:
                obj[path[-1]] = val
            return
        cur = scope.get(name)
        ex = Expr(lhs[1:], self, scope)
        args = ex.parse_args(cur if isinstance(cur, np.ndarray) else np.zeros((0, 0)))
        scope[name] = index_set(cur if isinstance(cur, np.ndarray) else None, args, val)


def run(name, *args, nout=1, mdir=MDIR_DEFAULT):
    """Execute ``<mdir>/<name>.m`` with the given arguments (numpy arrays / dict structs / floats)."""
    interp = Interp(mdir)

    def conv(a):
        if isinstance(a, dict):
            return {k: conv(v) for k, v in a.items()}
        if isinstance(a, str):
            return a
        return A(a)
    outs = interp.call(name, [conv(a) for a in args], nout)
    return outs if nout > 1 else outs[0]
