"""Plan-node plugins of the filter -> join -> group-by path and the operators either side of it."""
from . import (aggregate, cross_join, explain, filter, join, limit, project, sort, subquery_alias,  # noqa: A004
               table_scan, window)

DaskTableScanPlugin = table_scan.DaskTableScanPlugin
DaskFilterPlugin = filter.DaskFilterPlugin
DaskProjectPlugin = project.DaskProjectPlugin
DaskJoinPlugin = join.DaskJoinPlugin
DaskCrossJoinPlugin = cross_join.DaskCrossJoinPlugin
DaskAggregatePlugin = aggregate.DaskAggregatePlugin
DaskSortPlugin = sort.DaskSortPlugin
DaskLimitPlugin = limit.DaskLimitPlugin
SubqueryAlias = subquery_alias.SubqueryAlias
ExplainPlugin = explain.ExplainPlugin
DaskWindowPlugin = window.DaskWindowPlugin

ALL_PLUGINS = (DaskTableScanPlugin, DaskFilterPlugin, DaskProjectPlugin, DaskJoinPlugin, DaskCrossJoinPlugin,
               DaskAggregatePlugin, DaskSortPlugin, DaskLimitPlugin, SubqueryAlias, ExplainPlugin, DaskWindowPlugin)
