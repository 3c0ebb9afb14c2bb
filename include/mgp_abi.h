/*
 * mgp_abi.h -- the slice of Memgraph's query-module C ABI that the PageRank drop-in uses.
 *
 * Written from scratch as DECLARATIONS ONLY: the authoritative definition is the reference's
 * include/mg_procedure.h (2170 lines; memgraph/memgraph @ 292f896a).  Every prototype below names
 * the line of that header it restates, so a maintainer can diff them; the module also compiles
 * against the reference header itself (-DMGB200_USE_REFERENCE_MGP_HEADER -I<reference>/include),
 * and tests/test_module_host.py::test_mgp_abi_matches_the_reference_header checks every prototype,
 * enumerator and layout below against what the reference header gives (recorded under tests/golden/).
 *
 * Exports the module must provide (mg_procedure.h:1780-1793, loader: src/query/procedure/module.cpp:868-929):
 *     int mgp_init_module(struct mgp_module *, struct mgp_memory *);   required, 0 = success
 *     int mgp_shutdown_module(void);                                   optional
 * Imports (resolved against the host executable's dynamic symbol table, include/mg_procedure.syms):
 *     exactly the 30 functions the reference pagerank.so imports (SURVEY 8b) -- declared strong --
 *     plus three OPTIONAL ones declared weak, so the module still loads on a host lacking them:
 *     mgp_must_abort, mgp_result_reserve, mgp_log.
 */
#ifndef MGB200_MGP_ABI_H
#define MGB200_MGP_ABI_H

#ifdef MGB200_USE_REFERENCE_MGP_HEADER
#include "mg_procedure.h" /* the reference's own header, for the contract check */
#else

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#define MGP_ABI_ENUM enum class
#else
#define MGP_ABI_ENUM enum
#endif

/* mg_procedure.h:39-54 -- every fallible call returns one of these; results come back through the
 * trailing out-pointer. */
MGP_ABI_ENUM mgp_error{
    MGP_ERROR_NO_ERROR,            /* 0  */
    MGP_ERROR_UNKNOWN_ERROR,       /* 1  */
    MGP_ERROR_UNABLE_TO_ALLOCATE,  /* 2  */
    MGP_ERROR_INSUFFICIENT_BUFFER, /* 3  */
    MGP_ERROR_OUT_OF_RANGE,        /* 4  */
    MGP_ERROR_LOGIC_ERROR,         /* 5  */
    MGP_ERROR_DELETED_OBJECT,      /* 6  */
    MGP_ERROR_INVALID_ARGUMENT,    /* 7  */
    MGP_ERROR_KEY_ALREADY_EXISTS,  /* 8  */
    MGP_ERROR_IMMUTABLE_OBJECT,    /* 9  */
    MGP_ERROR_VALUE_CONVERSION,    /* 10 */
    MGP_ERROR_SERIALIZATION_ERROR, /* 11 */
    MGP_ERROR_AUTHORIZATION_ERROR, /* 12 */
    MGP_ERROR_NOT_YET_IMPLEMENTED, /* 13 */
};

/* opaque host objects (mg_procedure.h:84,129,155-167,708-710,779,1155,1707,1786-1789) */
struct mgp_memory;
struct mgp_graph;
struct mgp_value;
struct mgp_list;
struct mgp_vertex;
struct mgp_edge;
struct mgp_result;
struct mgp_result_record;
struct mgp_edges_iterator;
struct mgp_vertices_iterator;
struct mgp_type;
struct mgp_module;
struct mgp_proc;

struct mgp_vertex_id { /* :785-787, valid for one query execution */
  int64_t as_int;
};

MGP_ABI_ENUM mgp_log_level{ /* :1805-1812 */
    MGP_LOG_LEVEL_TRACE, MGP_LOG_LEVEL_DEBUG, MGP_LOG_LEVEL_INFO,
    MGP_LOG_LEVEL_WARN,  MGP_LOG_LEVEL_ERROR, MGP_LOG_LEVEL_CRITICAL,
};

MGP_ABI_ENUM mgp_value_type{ /* :197-217 (cugraph stand-in modules only: edge-property type test) */
    MGP_VALUE_TYPE_NULL, MGP_VALUE_TYPE_BOOL, MGP_VALUE_TYPE_INT, MGP_VALUE_TYPE_DOUBLE, MGP_VALUE_TYPE_STRING,
    MGP_VALUE_TYPE_LIST, MGP_VALUE_TYPE_MAP, MGP_VALUE_TYPE_VERTEX, MGP_VALUE_TYPE_EDGE, MGP_VALUE_TYPE_PATH,
    MGP_VALUE_TYPE_DATE, MGP_VALUE_TYPE_LOCAL_TIME, MGP_VALUE_TYPE_LOCAL_DATE_TIME, MGP_VALUE_TYPE_DURATION,
    MGP_VALUE_TYPE_ZONED_DATE_TIME, MGP_VALUE_TYPE_POINT_2D, MGP_VALUE_TYPE_POINT_3D, MGP_VALUE_TYPE_ENUM,
};

/* the procedure entry point (:1819): args, graph, result, memory live only during the call */
typedef void (*mgp_proc_cb)(struct mgp_list *, struct mgp_graph *, struct mgp_result *, struct mgp_memory *);

/* ---- values and argument list ---- */
void mgp_value_destroy(struct mgp_value *val);                                                          /* :222 */
enum mgp_error mgp_value_make_int(int64_t val, struct mgp_memory *memory, struct mgp_value **result);   /* :238 */
enum mgp_error mgp_value_make_double(double val, struct mgp_memory *memory, struct mgp_value **result); /* :243 */
enum mgp_error mgp_value_make_vertex(struct mgp_vertex *val, struct mgp_value **result); /* :272 takes ownership */
enum mgp_error mgp_value_get_int(struct mgp_value *val, int64_t *result);                               /* :436 */
enum mgp_error mgp_value_get_double(struct mgp_value *val, double *result);                             /* :441 */
enum mgp_error mgp_list_at(struct mgp_list *list, size_t index, struct mgp_value **result); /* :563 borrowed */
enum mgp_error mgp_value_get_vertex(struct mgp_value *val, struct mgp_vertex **result);     /* :461 borrowed; gpu_bfs only */

/* cugraph stand-in modules only (cugraph.pagerank.so, cugraph.personalized_pagerank.so): */
enum mgp_error mgp_value_make_string(const char *val, struct mgp_memory *memory, struct mgp_value **result); /* :248 */
enum mgp_error mgp_value_get_type(struct mgp_value *val, enum mgp_value_type *result);                       /* :353 */
enum mgp_error mgp_value_get_string(struct mgp_value *val, const char **result);               /* :446 borrowed */
enum mgp_error mgp_value_get_list(struct mgp_value *val, struct mgp_list **result);            /* :451 borrowed */
enum mgp_error mgp_list_size(struct mgp_list *list, size_t *result);                                         /* :554 */
enum mgp_error mgp_edge_get_property(struct mgp_edge *e, const char *property_name, struct mgp_memory *memory,
                                     struct mgp_value **result); /* :967 new value, Null when absent */
enum mgp_error mgp_type_string(struct mgp_type **result);                                                    /* :1692 */
enum mgp_error mgp_type_list(struct mgp_type *element_type, struct mgp_type **result);                       /* :1741 */

/* ---- result rows ---- */
enum mgp_error mgp_result_set_error_msg(struct mgp_result *res, const char *error_msg);                 /* :716 */
enum mgp_error mgp_result_new_record(struct mgp_result *res, struct mgp_result_record **result);        /* :721 */
enum mgp_error mgp_result_record_insert(struct mgp_result_record *record, const char *field_name,
                                        struct mgp_value *val); /* :731 copies val */

/* ---- graph iteration ---- */
void mgp_edges_iterator_destroy(struct mgp_edges_iterator *it);                                         /* :782 */
enum mgp_error mgp_vertex_get_id(struct mgp_vertex *v, struct mgp_vertex_id *result);                   /* :790 */
enum mgp_error mgp_vertex_iter_out_edges(struct mgp_vertex *v, struct mgp_memory *memory,
                                         struct mgp_edges_iterator **result);                           /* :901 */
enum mgp_error mgp_edges_iterator_get(struct mgp_edges_iterator *it, struct mgp_edge **result);         /* :913 */
enum mgp_error mgp_edges_iterator_next(struct mgp_edges_iterator *it, struct mgp_edge **result);        /* :920 */
enum mgp_error mgp_edge_get_to(struct mgp_edge *e, struct mgp_vertex **result);           /* :961 borrowed */
enum mgp_error mgp_graph_get_vertex_by_id(struct mgp_graph *g, struct mgp_vertex_id id, struct mgp_memory *memory,
                                          struct mgp_vertex **result); /* :1001 owned, NULL if absent */
enum mgp_error mgp_graph_is_transactional(struct mgp_graph *graph, int *result);                        /* :1120 */
void mgp_vertices_iterator_destroy(struct mgp_vertices_iterator *it);                                   /* :1158 */
enum mgp_error mgp_graph_iter_vertices(struct mgp_graph *g, struct mgp_memory *memory,
                                       struct mgp_vertices_iterator **result);                          /* :1163 */
enum mgp_error mgp_vertices_iterator_get(struct mgp_vertices_iterator *it, struct mgp_vertex **result); /* :1175 */
enum mgp_error mgp_graph_approximate_vertex_count(struct mgp_graph *graph, size_t *result);             /* :1178 */
enum mgp_error mgp_graph_approximate_edge_count(struct mgp_graph *graph, size_t *result);               /* :1181 */
enum mgp_error mgp_vertices_iterator_next(struct mgp_vertices_iterator *it, struct mgp_vertex **result); /* :1665 */

/* ---- type system and registration ---- */
enum mgp_error mgp_type_int(struct mgp_type **result);                                                  /* :1696 */
enum mgp_error mgp_type_float(struct mgp_type **result);                                                /* :1700 */
enum mgp_error mgp_type_node(struct mgp_type **result);                                                 /* :1725 */
enum mgp_error mgp_module_add_read_procedure(struct mgp_module *module, const char *name, mgp_proc_cb cb,
                                             struct mgp_proc **result);                                 /* :1838 */
enum mgp_error mgp_proc_add_arg(struct mgp_proc *proc, const char *name, struct mgp_type *type); /* :1890 gpu_bfs only */
enum mgp_error mgp_proc_add_opt_arg(struct mgp_proc *proc, const char *name, struct mgp_type *type,
                                    struct mgp_value *default_value); /* :1914 default is copied */
enum mgp_error mgp_proc_add_result(struct mgp_proc *proc, const char *name, struct mgp_type *type);     /* :1928 */

/* ---- optional (weak): absent on a minimal host => NULL, checked before use ---- */
#if defined(__GNUC__)
#define MGP_ABI_WEAK __attribute__((weak))
#else
#define MGP_ABI_WEAK
#endif
MGP_ABI_WEAK enum mgp_error mgp_result_reserve(struct mgp_result *res, size_t n);                       /* :725 */
MGP_ABI_WEAK enum mgp_error mgp_log(enum mgp_log_level log_level, const char *output);                  /* :1941 */
MGP_ABI_WEAK int mgp_must_abort(struct mgp_graph *graph);                                               /* :1962 */

#ifdef __cplusplus
}
#endif
#endif /* MGB200_USE_REFERENCE_MGP_HEADER */
#endif /* MGB200_MGP_ABI_H */
