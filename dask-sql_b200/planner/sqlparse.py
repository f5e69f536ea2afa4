"""SQL text -> syntax tree for the hot-path grammar.

The reference parses with sqlparser-rs 0.38 inside its Rust crate (src/parser.rs, src/sql.rs:570);
that crate cannot be built here (no rustc/cargo), so this is a small recursive-descent parser for

  [WITH name AS (select) [, ...]]
  SELECT [DISTINCT] item [, ...] FROM source [join ...] [WHERE e] [GROUP BY e, ...] [HAVING e]
  [ORDER BY e [ASC|DESC] [NULLS FIRST|LAST], ...] [LIMIT n [OFFSET m]]

  source := table [[AS] alias] | ( select ) [AS] alias
  join   := [INNER | LEFT [OUTER] | RIGHT [OUTER] | FULL [OUTER] | CROSS] JOIN source [ON e]

Expressions: literals, [qualifier.]column, + - * / %, comparisons, AND OR NOT, IS [NOT] NULL,
[NOT] BETWEEN, [NOT] IN (list), CAST(e AS type), CASE WHEN, function calls incl. aggregates with
DISTINCT and FILTER (WHERE ...), and window calls

  f(args) OVER ([PARTITION BY e, ...] [ORDER BY e [ASC|DESC] [NULLS FIRST|LAST], ...]
                [{ROWS | RANGE} {BETWEEN bound AND bound | bound}])
  bound  := UNBOUNDED PRECEDING | n PRECEDING | CURRENT ROW | n FOLLOWING | UNBOUNDED FOLLOWING

OVER / PARTITION / ROWS / RANGE / PRECEDING / FOLLOWING / UNBOUNDED / CURRENT / ROW are contextual
words as well: OVER starts a window only directly after a call's ")" and before "(", so columns and
aliases called over, rows, range or row keep parsing as before.

Statements around the path (custom statements of the reference's parser, src/parser.rs):
  CREATE [OR REPLACE] TABLE|VIEW [IF NOT EXISTS] [schema.]name AS [(] query [)]
  CREATE [OR REPLACE] TABLE [IF NOT EXISTS] [schema.]name WITH (key = literal [, ...])
  DROP TABLE [IF EXISTS] [schema.]name
CREATE / DROP / TABLE / VIEW / IF / EXISTS / REPLACE are contextual words, not reserved.
"""
import re
from typing import List, Optional

from ..utils import ParsingException

_TOKEN = re.compile(r"""
    (?P<ws>\s+|--[^\n]*)
  | (?P<num>(?:\d+\.\d*|\.\d+|\d+)(?:[eE][+-]?\d+)?)
  | (?P<str>'(?:[^']|'')*')
  | (?P<qid>"(?:[^"]|"")*"|`[^`]*`)
  | (?P<id>[A-Za-z_][A-Za-z_0-9$]*)
  | (?P<op><>|!=|<=|>=|\|\||[-+*/%=<>(),.;])
""", re.X)

KEYWORDS = {"SELECT", "FROM", "WHERE", "GROUP", "BY", "HAVING", "ORDER", "LIMIT", "OFFSET", "AS", "AND", "OR",
            "NOT", "IS", "NULL", "IN", "BETWEEN", "JOIN", "INNER", "LEFT", "RIGHT", "FULL", "OUTER", "CROSS", "ON",
            "DISTINCT", "CASE", "WHEN", "THEN", "ELSE", "END", "CAST", "TRUE", "FALSE", "ASC", "DESC", "NULLS",
            "FIRST", "LAST", "WITH", "FILTER", "UNION", "ALL", "EXPLAIN", "SEMI", "ANTI", "USING"}


class Tok:
    __slots__ = ("kind", "val", "pos")

    def __init__(self, kind, val, pos):
        self.kind, self.val, self.pos = kind, val, pos

    def __repr__(self):
        return f"{self.kind}:{self.val}"


def tokenize(sql: str) -> List[Tok]:
    out, pos = [], 0
    while pos < len(sql):
        m = _TOKEN.match(sql, pos)
        if not m:
            raise ParsingException(sql, f"Unexpected character {sql[pos]!r} at position {pos}")
        pos = m.end()
        if m.lastgroup == "ws":
            continue
        v = m.group(m.lastgroup)
        if m.lastgroup == "id":
            up = v.upper()
            out.append(Tok("kw", up, m.start()) if up in KEYWORDS else Tok("id", v, m.start()))
        elif m.lastgroup == "qid":
            out.append(Tok("id", v[1:-1].replace('""', '"'), m.start()))
        elif m.lastgroup == "str":
            out.append(Tok("str", v[1:-1].replace("''", "'"), m.start()))
        else:
            out.append(Tok(m.lastgroup, v, m.start()))
    out.append(Tok("eof", "", len(sql)))
    return out


class Node(dict):
    """Syntax-tree node: a dict with attribute access."""
    __getattr__ = dict.get

    def __init__(self, kind, **kw):
        super().__init__(kind=kind, **kw)


class Parser:
    def __init__(self, sql: str):
        self.sql = sql
        self.toks = tokenize(sql)
        self.i = 0

    # -- helpers
    @property
    def cur(self) -> Tok:
        return self.toks[self.i]

    def error(self, msg):
        raise ParsingException(self.sql, f"{msg} near position {self.cur.pos}: ...{self.sql[self.cur.pos:self.cur.pos + 30]!r}")

    def at_kw(self, *kws):
        return self.cur.kind == "kw" and self.cur.val in kws

    def at_op(self, *ops):
        return self.cur.kind == "op" and self.cur.val in ops

    def eat_kw(self, *kws):
        if self.at_kw(*kws):
            self.i += 1
            return self.toks[self.i - 1].val
        return None

    def eat_op(self, *ops):
        if self.at_op(*ops):
            self.i += 1
            return self.toks[self.i - 1].val
        return None

    def expect_kw(self, kw):
        if not self.eat_kw(kw):
            self.error(f"Expected {kw}")

    def expect_op(self, op):
        if not self.eat_op(op):
            self.error(f"Expected '{op}'")

    def ident(self):
        if self.cur.kind == "id":
            self.i += 1
            return self.toks[self.i - 1].val
        # non-reserved use of some keywords as identifiers (e.g. a column called "first")
        if self.cur.kind == "kw" and self.cur.val in ("FIRST", "LAST", "FILTER", "ALL"):
            self.i += 1
            return self.toks[self.i - 1].val.lower()
        self.error("Expected identifier")

    def at_word(self, *words):
        return self.cur.kind == "id" and self.cur.val.upper() in words

    def eat_word(self, *words):
        if self.at_word(*words):
            self.i += 1
            return self.toks[self.i - 1].val.upper()
        return None

    def expect_word(self, word):
        if not self.eat_word(word):
            self.error(f"Expected {word}")

    def qualified_name(self) -> str:
        parts = [self.ident()]
        while self.eat_op("."):
            parts.append(self.ident())
        return ".".join(parts)

    # -- statements
    def parse_ddl(self) -> Optional[Node]:
        if self.at_word("DROP") and self.toks[self.i + 1].kind == "id":
            self.i += 1
            self.expect_word("TABLE")
            if_exists = False
            if self.at_word("IF"):
                self.i += 1
                self.expect_word("EXISTS")
                if_exists = True
            return Node("drop_table", name=self.qualified_name(), if_exists=if_exists)
        if not (self.at_word("CREATE") and self.toks[self.i + 1].kind in ("id", "kw")):
            return None
        self.i += 1
        or_replace = False
        if self.eat_kw("OR"):
            self.expect_word("REPLACE")
            or_replace = True
        what = self.eat_word("TABLE", "VIEW")
        if what is None:
            self.error("Expected TABLE or VIEW")
        if_not_exists = False
        if self.at_word("IF"):
            self.i += 1
            self.expect_kw("NOT")
            self.expect_word("EXISTS")
            if_not_exists = True
        name = self.qualified_name()
        if self.eat_kw("AS"):
            paren = bool(self.at_op("(") and self.toks[self.i + 1].kind == "kw"
                         and self.toks[self.i + 1].val in ("SELECT", "WITH") and self.eat_op("("))
            q = self.parse_query()
            if paren:
                self.expect_op(")")
            return Node("create_memory_table", name=name, query=q, or_replace=or_replace,
                        if_not_exists=if_not_exists, is_table=(what == "TABLE"))
        if what == "TABLE" and self.eat_kw("WITH"):
            self.expect_op("(")
            kwargs = {}
            while True:
                key = self.ident()
                self.expect_op("=")
                lit = self.parse_primary()
                neg = False
                if lit.kind != "lit":
                    self.error("Expected a literal value")
                kwargs[key] = lit.value
                if not self.eat_op(","):
                    break
            self.expect_op(")")
            return Node("create_table", name=name, kwargs=kwargs, or_replace=or_replace, if_not_exists=if_not_exists)
        self.error("Expected AS or WITH")

    def parse_statement(self) -> Node:
        ddl = self.parse_ddl()
        if ddl is not None:
            self.eat_op(";")
            if self.cur.kind != "eof":
                self.error("Unexpected trailing input")
            return ddl
        explain = bool(self.eat_kw("EXPLAIN"))
        q = self.parse_query()
        self.eat_op(";")
        if self.cur.kind != "eof":
            self.error("Unexpected trailing input")
        if explain:
            return Node("explain", query=q)
        return q

    def parse_query(self) -> Node:
        ctes = []
        if self.eat_kw("WITH"):
            while True:
                name = self.ident()
                self.expect_kw("AS")
                self.expect_op("(")
                ctes.append((name, self.parse_query()))
                self.expect_op(")")
                if not self.eat_op(","):
                    break
        q = self.parse_select()
        q["ctes"] = ctes
        return q

    def parse_select(self) -> Node:
        self.expect_kw("SELECT")
        distinct = bool(self.eat_kw("DISTINCT"))
        self.eat_kw("ALL")
        items = [self.parse_select_item()]
        while self.eat_op(","):
            items.append(self.parse_select_item())
        source = None
        if self.eat_kw("FROM"):
            source = self.parse_from()
        where = self.parse_expr() if self.eat_kw("WHERE") else None
        group_by = []
        if self.eat_kw("GROUP"):
            self.expect_kw("BY")
            group_by.append(self.parse_expr())
            while self.eat_op(","):
                group_by.append(self.parse_expr())
        having = self.parse_expr() if self.eat_kw("HAVING") else None
        order_by = []
        if self.eat_kw("ORDER"):
            self.expect_kw("BY")
            order_by = self.parse_order_items()
        limit = offset = None
        if self.eat_kw("LIMIT"):
            limit = self.parse_expr()
        if self.eat_kw("OFFSET"):
            offset = self.parse_expr()
        return Node("select", distinct=distinct, items=items, source=source, where=where, group_by=group_by,
                    having=having, order_by=order_by, limit=limit, offset=offset, ctes=[])

    def parse_order_items(self):
        """e [ASC|DESC] [NULLS FIRST|LAST], ... -> [(e, asc, nulls_first or None)]"""
        items = []
        while True:
            e = self.parse_expr()
            asc = True
            if self.eat_kw("DESC"):
                asc = False
            else:
                self.eat_kw("ASC")
            nulls_first = None
            if self.eat_kw("NULLS"):
                nulls_first = bool(self.eat_kw("FIRST"))
                if not nulls_first:
                    self.expect_kw("LAST")
            items.append((e, asc, nulls_first))
            if not self.eat_op(","):
                return items

    def parse_window_spec(self) -> Node:
        """The parenthesised part after OVER (the opening "(" is consumed)."""
        partition, order, frame = [], [], None
        if self.eat_word("PARTITION"):
            self.expect_kw("BY")
            partition.append(self.parse_expr())
            while self.eat_op(","):
                partition.append(self.parse_expr())
        if self.eat_kw("ORDER"):
            self.expect_kw("BY")
            order = self.parse_order_items()
        unit = self.eat_word("ROWS", "RANGE")
        if unit:
            if self.eat_kw("BETWEEN"):
                lo = self.parse_frame_bound()
                self.expect_kw("AND")
                hi = self.parse_frame_bound()
            else:                               # "ROWS 3 PRECEDING" = BETWEEN 3 PRECEDING AND CURRENT ROW
                lo, hi = self.parse_frame_bound(), ("CURRENT", 0)
            frame = (unit, lo, hi)
        self.expect_op(")")
        return Node("window", partition=partition, order=order, frame=frame)

    def parse_frame_bound(self):
        """-> (kind, offset), kind in UNBOUNDED_PRECEDING | PRECEDING | CURRENT | FOLLOWING | UNBOUNDED_FOLLOWING"""
        if self.eat_word("UNBOUNDED"):
            d = self.eat_word("PRECEDING", "FOLLOWING")
            if d is None:
                self.error("Expected PRECEDING or FOLLOWING")
            return ("UNBOUNDED_" + d, None)
        if self.eat_word("CURRENT"):
            self.expect_word("ROW")
            return ("CURRENT", 0)
        t = self.cur
        if t.kind == "num":
            self.i += 1
            d = self.eat_word("PRECEDING", "FOLLOWING")
            if d is None:
                self.error("Expected PRECEDING or FOLLOWING")
            if not re.fullmatch(r"\d+", t.val):
                return (d, float(t.val))          # rejected by the binder with a clear message
            return (d, int(t.val))
        self.error("Expected a window frame bound")

    def parse_select_item(self):
        if self.eat_op("*"):
            return (Node("star", qualifier=None), None)
        # qualifier.*
        if self.cur.kind == "id" and self.toks[self.i + 1].kind == "op" and self.toks[self.i + 1].val == "." \
                and self.toks[self.i + 2].kind == "op" and self.toks[self.i + 2].val == "*":
            q = self.ident()
            self.i += 2
            return (Node("star", qualifier=q), None)
        e = self.parse_expr()
        alias = None
        if self.eat_kw("AS"):
            alias = self.ident()
        elif self.cur.kind == "id":
            alias = self.ident()
        return (e, alias)

    def parse_from(self) -> Node:
        left = self.parse_source()
        while True:
            if self.eat_op(","):
                right = self.parse_source()
                left = Node("join", left=left, right=right, how="CROSS", on=None)
                continue
            how = None
            if self.eat_kw("INNER"):
                how = "INNER"
            elif self.eat_kw("LEFT"):
                how = "LEFT"
                if self.eat_kw("SEMI"):
                    how = "LEFTSEMI"
                elif self.eat_kw("ANTI"):
                    how = "LEFTANTI"
                else:
                    self.eat_kw("OUTER")
            elif self.eat_kw("RIGHT"):
                how = "RIGHT"
                self.eat_kw("OUTER")
            elif self.eat_kw("FULL"):
                how = "FULL"
                self.eat_kw("OUTER")
            elif self.eat_kw("CROSS"):
                how = "CROSS"
            if how is None and not self.at_kw("JOIN"):
                return left
            self.expect_kw("JOIN")
            right = self.parse_source()
            on = None
            if self.eat_kw("ON"):
                on = self.parse_expr()
            elif self.eat_kw("USING"):
                self.expect_op("(")
                cols = [self.ident()]
                while self.eat_op(","):
                    cols.append(self.ident())
                self.expect_op(")")
                on = Node("using", cols=cols)
            left = Node("join", left=left, right=right, how=how or "INNER", on=on)

    def parse_source(self) -> Node:
        if self.eat_op("("):
            q = self.parse_query()
            self.expect_op(")")
            self.eat_kw("AS")
            alias = self.ident()
            return Node("subquery", query=q, alias=alias)
        parts = [self.ident()]
        while self.eat_op("."):
            parts.append(self.ident())
        alias = None
        if self.eat_kw("AS"):
            alias = self.ident()
        elif self.cur.kind == "id":
            alias = self.ident()
        return Node("table", name=parts, alias=alias)

    # -- expressions (precedence climbing)
    def parse_expr(self) -> Node:
        return self.parse_or()

    def parse_or(self):
        e = self.parse_and()
        while self.eat_kw("OR"):
            e = Node("bin", op="OR", l=e, r=self.parse_and())
        return e

    def parse_and(self):
        e = self.parse_not()
        while self.eat_kw("AND"):
            e = Node("bin", op="AND", l=e, r=self.parse_not())
        return e

    def parse_not(self):
        if self.eat_kw("NOT"):
            return Node("not", e=self.parse_not())
        return self.parse_cmp()

    def parse_cmp(self):
        e = self.parse_add()
        while True:
            if self.at_op("=", "<>", "!=", "<", "<=", ">", ">="):
                op = self.eat_op("=", "<>", "!=", "<", "<=", ">", ">=")
                e = Node("bin", op="!=" if op == "<>" else op, l=e, r=self.parse_add())
            elif self.at_kw("IS"):
                self.i += 1
                neg = bool(self.eat_kw("NOT"))
                if self.eat_kw("NULL"):
                    e = Node("isnull", e=e, negated=neg)
                elif self.eat_kw("TRUE"):
                    e = Node("istrue", e=e, negated=neg, value=True)
                elif self.eat_kw("FALSE"):
                    e = Node("istrue", e=e, negated=neg, value=False)
                elif self.eat_word("UNKNOWN"):      # a boolean is UNKNOWN iff it is NULL (call.py:1123-1124)
                    e = Node("isnull", e=e, negated=neg)
                else:
                    self.error("Expected NULL, TRUE, FALSE or UNKNOWN after IS")
            elif self.at_kw("NOT") and self.toks[self.i + 1].kind == "kw" and self.toks[self.i + 1].val in ("BETWEEN", "IN"):
                self.i += 1
                e = self._between_or_in(e, True)
            elif self.at_kw("BETWEEN", "IN"):
                e = self._between_or_in(e, False)
            else:
                return e

    def _between_or_in(self, e, negated):
        if self.eat_kw("BETWEEN"):
            lo = self.parse_add()
            self.expect_kw("AND")
            hi = self.parse_add()
            return Node("between", e=e, lo=lo, hi=hi, negated=negated)
        self.expect_kw("IN")
        self.expect_op("(")
        if self.at_kw("SELECT", "WITH"):
            self.error("IN (subquery) is outside the hot-path grammar")
        items = [self.parse_expr()]
        while self.eat_op(","):
            items.append(self.parse_expr())
        self.expect_op(")")
        return Node("inlist", e=e, items=items, negated=negated)

    def parse_add(self):
        e = self.parse_mul()
        while self.at_op("+", "-"):
            op = self.eat_op("+", "-")
            e = Node("bin", op=op, l=e, r=self.parse_mul())
        return e

    def parse_mul(self):
        e = self.parse_unary()
        while self.at_op("*", "/", "%"):
            op = self.eat_op("*", "/", "%")
            e = Node("bin", op=op, l=e, r=self.parse_unary())
        return e

    def parse_unary(self):
        if self.eat_op("-"):
            inner = self.parse_unary()
            if inner.kind == "lit" and isinstance(inner.value, (int, float)) and not isinstance(inner.value, bool):
                return Node("lit", value=-inner.value)
            return Node("neg", e=inner)
        if self.eat_op("+"):
            return self.parse_unary()
        return self.parse_primary()

    def parse_primary(self):
        t = self.cur
        if t.kind == "num":
            self.i += 1
            txt = t.val
            if re.fullmatch(r"\d+", txt):
                return Node("lit", value=int(txt))
            return Node("lit", value=float(txt))
        if t.kind == "str":
            self.i += 1
            return Node("lit", value=t.val)
        if self.eat_kw("TRUE"):
            return Node("lit", value=True)
        if self.eat_kw("FALSE"):
            return Node("lit", value=False)
        if self.eat_kw("NULL"):
            return Node("lit", value=None)
        if self.eat_op("("):
            e = self.parse_expr()
            self.expect_op(")")
            return e
        if self.eat_kw("CAST"):
            self.expect_op("(")
            e = self.parse_expr()
            self.expect_kw("AS")
            ty = self.ident()
            if ty.upper() == "DOUBLE" and self.cur.kind == "id" and self.cur.val.upper() == "PRECISION":
                self.i += 1
            if self.eat_op("("):  # DECIMAL(p, s) and friends
                while not self.eat_op(")"):
                    self.i += 1
            self.expect_op(")")
            return Node("cast", e=e, type=ty.upper())
        if self.eat_kw("CASE"):
            operand = None
            if not self.at_kw("WHEN"):
                operand = self.parse_expr()
            whens = []
            while self.eat_kw("WHEN"):
                w = self.parse_expr()
                self.expect_kw("THEN")
                whens.append((Node("bin", op="=", l=operand, r=w) if operand is not None else w, self.parse_expr()))
            other = self.parse_expr() if self.eat_kw("ELSE") else None
            self.expect_kw("END")
            return Node("case", whens=whens, other=other)
        if t.kind == "id" or (t.kind == "kw" and t.val in ("LEFT", "RIGHT", "FIRST", "LAST", "FILTER")
                              and self.toks[self.i + 1].kind == "op" and self.toks[self.i + 1].val in ("(", ".")):
            name = self.ident() if t.kind == "id" else (self.toks[self.i].val, setattr(self, "i", self.i + 1))[0]
            if self.eat_op("("):  # function call
                distinct = bool(self.eat_kw("DISTINCT"))
                args, star = [], False
                if self.eat_op("*"):
                    star = True
                elif not self.at_op(")"):
                    args.append(self.parse_expr())
                    while self.eat_op(","):
                        args.append(self.parse_expr())
                self.expect_op(")")
                filt = None
                if self.at_kw("FILTER") and self.toks[self.i + 1].kind == "op" and self.toks[self.i + 1].val == "(":
                    self.i += 2
                    self.expect_kw("WHERE")
                    filt = self.parse_expr()
                    self.expect_op(")")
                over = None
                if self.at_word("OVER") and self.toks[self.i + 1].kind == "op" and self.toks[self.i + 1].val == "(":
                    self.i += 2
                    over = self.parse_window_spec()
                return Node("func", name=name.upper(), args=args, distinct=distinct, star=star, filter=filt, over=over)
            parts = [name]
            while self.eat_op("."):
                parts.append(self.ident())
            return Node("col", parts=parts)
        self.error("Unexpected token")


def parse_sql(sql: str) -> Node:
    return Parser(sql).parse_statement()
