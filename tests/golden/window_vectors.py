"""Golden vectors for window functions, TRANSCRIBED from the reference's known-answer tests
(dask-contrib/dask-sql @ f186de3, tests/integration/test_over.py).  Kept apart from
reference_vectors.CASES so that the cases there keep exactly their meaning.  Every case cites the
reference test it comes from; `expected` is the literal frame of the reference test (its row order is
not part of the answer: the reference compares with check_index=False after sorting)."""
import numpy as np
import pandas as pd

from .reference_vectors import user_table_1, user_table_2


def tmp():                  # test_over.py:147-148
    return pd.DataFrame({"a": range(5)})


FIXTURES = {"user_table_1": user_table_1, "user_table_2": user_table_2, "tmp": tmp}

NaN = np.nan

CASES = [
    dict(name="over_with_sorting", cite="tests/integration/test_over.py:7-20", tables=["user_table_1"],
         sql='SELECT user_id, b, ROW_NUMBER() OVER (ORDER BY user_id, b) AS "R" FROM user_table_1',
         expected=pd.DataFrame({"user_id": [1, 2, 2, 3], "b": [3, 1, 3, 3], "R": [1, 2, 3, 4]})),
    dict(name="over_with_partitioning", cite="tests/integration/test_over.py:23-37", tables=["user_table_2"],
         sql='SELECT user_id, c, ROW_NUMBER() OVER (PARTITION BY c) AS "R" FROM user_table_2 ORDER BY user_id, c',
         expected=pd.DataFrame({"user_id": [1, 1, 2, 4], "c": [1, 2, 3, 4], "R": [1, 1, 1, 1]})),
    dict(name="over_with_grouping_and_sort", cite="tests/integration/test_over.py:40-53", tables=["user_table_1"],
         sql='SELECT user_id, b, ROW_NUMBER() OVER (PARTITION BY user_id ORDER BY b) AS "R" FROM user_table_1',
         expected=pd.DataFrame({"user_id": [1, 2, 2, 3], "b": [3, 1, 3, 3], "R": [1, 1, 2, 1]})),
    dict(name="over_with_different", cite="tests/integration/test_over.py:56-76", tables=["user_table_1"],
         sql='''SELECT user_id, b,
                       ROW_NUMBER() OVER (PARTITION BY user_id ORDER BY b) AS "R1",
                       ROW_NUMBER() OVER (ORDER BY user_id, b) AS "R2"
                FROM user_table_1''',
         expected=pd.DataFrame({"user_id": [2, 1, 2, 3], "b": [3, 3, 1, 3], "R1": [2, 1, 1, 1], "R2": [3, 1, 2, 4]})),
    # O3 is commented out in the reference test and pinned by its xfail test_over_single_value
    # (test_over.py:120-141) with the same answers as O2
    dict(name="over_calls", cite="tests/integration/test_over.py:81-117 (+ O3: :123-141)", tables=["user_table_1"],
         sql='''SELECT user_id, b,
                       ROW_NUMBER() OVER (PARTITION BY user_id ORDER BY b) AS "O1",
                       FIRST_VALUE(user_id*10 - b) OVER (PARTITION BY user_id ORDER BY b) AS "O2",
                       SINGLE_VALUE(user_id*10 - b) OVER (PARTITION BY user_id ORDER BY b) AS "O3",
                       LAST_VALUE(user_id*10 - b) OVER (PARTITION BY user_id ORDER BY b
                           ROWS BETWEEN UNBOUNDED PRECEDING AND UNBOUNDED FOLLOWING) AS "O4",
                       SUM(user_id) OVER (PARTITION BY user_id ORDER BY b) AS "O5",
                       AVG(user_id) OVER (PARTITION BY user_id ORDER BY b) AS "O6",
                       COUNT(*) OVER (PARTITION BY user_id ORDER BY b) AS "O7",
                       COUNT(b) OVER (PARTITION BY user_id ORDER BY b) AS "O7b",
                       MAX(b) OVER (PARTITION BY user_id ORDER BY b) AS "O8",
                       MIN(b) OVER (PARTITION BY user_id ORDER BY b) AS "O9"
                FROM user_table_1''',
         expected=pd.DataFrame({"user_id": [2, 1, 2, 3], "b": [3, 3, 1, 3], "O1": [2, 1, 1, 1], "O2": [19, 7, 19, 27],
                                "O3": [19, 7, 19, 27], "O4": [17, 7, 17, 27], "O5": [4, 1, 2, 3], "O6": [2, 1, 2, 3],
                                "O7": [2, 1, 1, 1], "O7b": [2, 1, 1, 1], "O8": [3, 3, 1, 3], "O9": [1, 3, 1, 3]})),
    dict(name="over_with_windows", cite="tests/integration/test_over.py:146-185", tables=["tmp"],
         sql='''SELECT a,
                    SUM(a) OVER (ORDER BY a ROWS BETWEEN 2 PRECEDING AND CURRENT ROW) AS "O1",
                    SUM(a) OVER (ORDER BY a ROWS BETWEEN 2 PRECEDING AND 3 FOLLOWING) AS "O2",
                    SUM(a) OVER (ORDER BY a ROWS BETWEEN 2 PRECEDING AND UNBOUNDED FOLLOWING) AS "O3",
                    SUM(a) OVER (ORDER BY a ROWS BETWEEN CURRENT ROW AND 3 FOLLOWING) AS "O4",
                    SUM(a) OVER (ORDER BY a ROWS BETWEEN CURRENT ROW AND UNBOUNDED FOLLOWING) AS "O5",
                    SUM(a) OVER (ORDER BY a ROWS BETWEEN UNBOUNDED PRECEDING AND CURRENT ROW) AS "O6",
                    SUM(a) OVER (ORDER BY a ROWS BETWEEN UNBOUNDED PRECEDING AND 3 FOLLOWING) AS "O7",
                    SUM(a) OVER (ORDER BY a ROWS BETWEEN UNBOUNDED PRECEDING AND UNBOUNDED FOLLOWING) AS "O8",
                    SUM(a) OVER (ORDER BY a ROWS BETWEEN 3 FOLLOWING AND 3 FOLLOWING) AS "O9",
                    COUNT(a) OVER (ORDER BY a ROWS BETWEEN 3 FOLLOWING AND 3 FOLLOWING) AS "O9a",
                    SUM(a) OVER (ORDER BY a ROWS BETWEEN 3 PRECEDING AND 1 PRECEDING) AS "O10"
                FROM tmp''',
         expected=pd.DataFrame({"a": [0, 1, 2, 3, 4], "O1": [0, 1, 3, 6, 9], "O2": [6, 10, 10, 10, 9],
                                "O3": [10, 10, 10, 10, 9], "O4": [6, 10, 9, 7, 4], "O5": [10, 10, 9, 7, 4],
                                "O6": [0, 1, 3, 6, 10], "O7": [6, 10, 10, 10, 10], "O8": [10, 10, 10, 10, 10],
                                "O9": [3, 4, NaN, NaN, NaN], "O9a": [1, 1, 0, 0, 0], "O10": [NaN, 0, 1, 3, 6]})),
]


def tables_of(case):
    return {t: FIXTURES[t]() for t in case["tables"]}
