"""The bluespot filter of `malstroem complete` / `malstroem bluespots` (`-filter`, bluespots.py:23-46 and
scripts/_utils.py:29-40) as a small postfix program that the device evaluates per label (csrc/bfilter.cu).

The CLI turns its filter text into `lambda stats: <text>` over three per-label numbers of the RAW bluespots:
`area` = cell count * cell area, `maxdepth` = the deepest depth, `volume` = the depth sum * cell area (numpy float64
scalars).  `compile_filter` accepts the part of Python's expression grammar that such a filter uses:

- the names `area`, `maxdepth`, `volume`; int, float and bool literals (ints up to 2**53 in magnitude);
- unary `-` / `+`, binary `+ - * /`, parentheses;
- comparisons `< <= > >= == !=` (chained ones too, `0.1 < maxdepth < 2`), `and`, `or`, `not`.

Comparisons and boolean operators may only stand in boolean context — the whole expression, or an operand of `and` /
`or` / `not` — and their operands must be arithmetic; in boolean context a number counts as true when it is != 0 (NaN
is true, as in Python).  Constant subexpressions are folded with Python's own arithmetic, so `1/0` fails here as it
would in the reference.  Everything else raises ValueError naming the offending node.

Every operation is one IEEE float64 operation on the device, so keep decisions are bitwise numpy's on the same
stats.  The stats themselves are the device's: `volume` thresholds decide on `st_sum`, whose float64 sum is
associated differently from the reference's raster-order sum (within 1e-6 relative), so a label whose volume lies
within that of a threshold may decide differently — as on the plug-in path.
"""
import ast
import operator

import numpy as np

from . import _lib

# op codes: the MS_BF_* enum of include/malstroem_b200.h
AREA, MAXDEPTH, VOLUME, CONST, NEG, NOT, ADD, SUB, MUL, DIV, LT, LE, GT, GE, EQ, NE, AND, OR = range(1, 19)
NAMES = {"area": AREA, "maxdepth": MAXDEPTH, "volume": VOLUME}
MAX_OPS, MAX_STACK = _lib.MS_BF_MAX_OPS, _lib.MS_BF_MAX_STACK
_INT_LIMIT = 2 ** 53

_ARITH = {ast.Add: (ADD, operator.add), ast.Sub: (SUB, operator.sub), ast.Mult: (MUL, operator.mul),
          ast.Div: (DIV, operator.truediv)}
_CMP = {ast.Lt: (LT, operator.lt), ast.LtE: (LE, operator.le), ast.Gt: (GT, operator.gt), ast.GtE: (GE, operator.ge),
        ast.Eq: (EQ, operator.eq), ast.NotEq: (NE, operator.ne)}
_SPELLING = {ast.Pow: "**", ast.Mod: "%", ast.FloorDiv: "//", ast.MatMult: "@", ast.LShift: "<<", ast.RShift: ">>",
             ast.BitOr: "|", ast.BitAnd: "&", ast.BitXor: "^", ast.Invert: "~", ast.Is: "is", ast.IsNot: "is not",
             ast.In: "in", ast.NotIn: "not in"}


class FilterProgram(object):
    """A compiled filter: `code` is a tuple of (op, immediate) pairs in postfix order."""

    def __init__(self, text, code):
        self.text, self.code = text, tuple(code)
        depth = self.max_stack = 0
        for op, _ in self.code:
            depth += 1 if op <= CONST else 0 if op <= NOT else -1
            self.max_stack = max(self.max_stack, depth)
        if len(self.code) > MAX_OPS or self.max_stack > MAX_STACK:
            raise ValueError("bluespot filter %r: %d operations and a stack of %d values exceed the device's %d / %d"
                             % (text, len(self.code), self.max_stack, MAX_OPS, MAX_STACK))
        self.reads = frozenset(op for op, _ in self.code if op in (AREA, MAXDEPTH, VOLUME))

    def struct(self, cell_area):
        """The C struct ms_bluespot_filter of this program and `cell_area`."""
        ca = float(cell_area)
        if not (ca > 0.0 and np.isfinite(ca)):
            raise ValueError("bluespot filter: cell_area must be finite and > 0 (%r)" % cell_area)
        f = _lib.MsBluespotFilter()
        f.n_ops = len(self.code)
        for k, (op, imm) in enumerate(self.code):
            f.op[k], f.imm[k] = op, imm
        f.cell_area = ca
        return f

    def evaluate(self, area, maxdepth, volume):
        """Keep decisions (bool array) of this program on float64 arrays (numpy or torch) of one shape; label 0 is
        not treated specially here.  The same operations as the device, element-wise."""
        def full(c):
            return np.full(area.shape, c, np.float64) if isinstance(area, np.ndarray) else area.new_full(area.shape, c)

        with np.errstate(all="ignore"):
            st = []
            for op, imm in self.code:
                if op <= CONST:
                    st.append({AREA: area, MAXDEPTH: maxdepth, VOLUME: volume}.get(op) if op != CONST else full(imm))
                elif op == NEG:
                    st[-1] = -st[-1]
                elif op == NOT:
                    st[-1] = ~(st[-1] != 0)
                else:
                    b = st.pop()
                    a = st.pop()
                    st.append({ADD: lambda: a + b, SUB: lambda: a - b, MUL: lambda: a * b, DIV: lambda: a / b,
                               LT: lambda: a < b, LE: lambda: a <= b, GT: lambda: a > b, GE: lambda: a >= b,
                               EQ: lambda: a == b, NE: lambda: a != b, AND: lambda: (a != 0) & (b != 0),
                               OR: lambda: (a != 0) | (b != 0)}[op]())
            return st[0] != 0

    def __repr__(self):
        return "FilterProgram(%r, %d ops)" % (self.text, len(self.code))


def compile_filter(text):
    """The CLI's filter text -> FilterProgram; None or "" -> None (no filter: every raw bluespot is kept)."""
    if text is None or text == "":
        return None
    if not isinstance(text, str):
        raise ValueError("bluespot filter: expected the filter text, got %s" % type(text).__name__)
    try:
        tree = ast.parse(text.strip(), mode="eval")
    except SyntaxError as e:
        raise ValueError("bluespot filter %r: syntax error: %s" % (text, e.msg)) from None
    c = _Compiler(text)
    return FilterProgram(text, c.emit(c.boolean(tree.body)))


class _Compiler(object):
    """Both methods return ("const", python value) for a constant subexpression or ("code", [(op, imm)...])."""

    def __init__(self, text):
        self.text = text

    def fail(self, node, what):
        raise ValueError("bluespot filter %r: %s (column %d)" % (self.text, what, getattr(node, "col_offset", 0)))

    def emit(self, r):
        kind, v = r
        return [(CONST, float(v))] if kind == "const" else v

    def const(self, node, v):
        if type(v) is int and abs(v) > _INT_LIMIT:
            self.fail(node, "integer %d is larger than 2**53 in magnitude" % v)
        return ("const", v)

    def arith(self, node):
        if isinstance(node, ast.Constant):
            if type(node.value) not in (bool, int, float):
                self.fail(node, "unsupported constant %r" % (node.value,))
            return self.const(node, node.value)
        if isinstance(node, ast.Name):
            if node.id not in NAMES:
                self.fail(node, "unknown name %r (allowed: area, maxdepth, volume)" % node.id)
            return ("code", [(NAMES[node.id], 0.0)])
        if isinstance(node, ast.UnaryOp):
            if isinstance(node.op, ast.Not):
                self.fail(node, "'not' is allowed only in boolean context, not as an arithmetic operand")
            if not isinstance(node.op, (ast.USub, ast.UAdd)):
                self.fail(node, "unsupported operator %r" % _SPELLING.get(type(node.op), type(node.op).__name__))
            kind, v = self.arith(node.operand)
            neg = isinstance(node.op, ast.USub)
            if kind == "const":
                return self.const(node, -v if neg else +v)
            return ("code", v + [(NEG, 0.0)] if neg else v)
        if isinstance(node, ast.BinOp):
            if type(node.op) not in _ARITH:
                self.fail(node, "unsupported operator %r" % _SPELLING.get(type(node.op), type(node.op).__name__))
            op, fn = _ARITH[type(node.op)]
            a, b = self.arith(node.left), self.arith(node.right)
            if a[0] == "const" and b[0] == "const":
                try:
                    return self.const(node, fn(a[1], b[1]))
                except ZeroDivisionError:
                    self.fail(node, "division by zero in a constant subexpression")
            return ("code", self.emit(a) + self.emit(b) + [(op, 0.0)])
        if isinstance(node, (ast.Compare, ast.BoolOp)):
            self.fail(node, "%s is allowed only in boolean context, not as an arithmetic operand"
                      % ("a comparison" if isinstance(node, ast.Compare) else "'and' / 'or'"))
        self.fail(node, "unsupported syntax %s" % type(node).__name__)

    def boolean(self, node):
        if isinstance(node, ast.BoolOp):
            op = AND if isinstance(node.op, ast.And) else OR
            parts = [self.boolean(v) for v in node.values]
            if all(k == "const" for k, _ in parts):
                truth = [bool(v) for _, v in parts]
                return ("const", all(truth) if op == AND else any(truth))
            code = self.emit(parts[0])
            for p in parts[1:]:
                code += self.emit(p) + [(op, 0.0)]
            return ("code", code)
        if isinstance(node, ast.UnaryOp) and isinstance(node.op, ast.Not):
            kind, v = self.boolean(node.operand)
            return ("const", not v) if kind == "const" else ("code", v + [(NOT, 0.0)])
        if isinstance(node, ast.Compare):
            terms = [self.arith(x) for x in [node.left] + list(node.comparators)]
            pairs = []
            for k, cop in enumerate(node.ops):
                if type(cop) not in _CMP:
                    self.fail(node, "unsupported comparison %r" % _SPELLING.get(type(cop), type(cop).__name__))
                op, fn = _CMP[type(cop)]
                a, b = terms[k], terms[k + 1]
                if a[0] == "const" and b[0] == "const":
                    pairs.append(("const", fn(a[1], b[1])))
                else:
                    pairs.append(("code", self.emit(a) + self.emit(b) + [(op, 0.0)]))
            if len(pairs) == 1:
                return pairs[0]
            return self.boolean_of(pairs)
        return self.arith(node)

    def boolean_of(self, pairs):
        """`and` over already compiled terms (a chained comparison)."""
        if all(k == "const" for k, _ in pairs):
            return ("const", all(bool(v) for _, v in pairs))
        code = self.emit(pairs[0])
        for p in pairs[1:]:
            code += self.emit(p) + [(AND, 0.0)]
        return ("code", code)


def label_ranges_after_filter(label_ranges, keep):
    """The (offset, count) label range of every band after a filter: the band that numbered a raw label still owns
    it, so (o, c) -> (kept[o], kept[o + c] - kept[o]) with kept[k] = kept labels among 1..k.  keep: bool sequence over
    the raw labels 0..nlabels (keep[0] ignored)."""
    k = np.asarray(keep, dtype=bool).copy()
    k[:1] = False
    kept = np.cumsum(k)
    return [(int(kept[o]), int(kept[o + c] - kept[o])) for o, c in label_ranges]
