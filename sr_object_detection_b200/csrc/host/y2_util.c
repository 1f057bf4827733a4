/*
 * Host utilities of the drop-in C API: error conventions, line/option/list helpers, label and
 * map readers, WordTree reader, CPU bilinear resize.  Behavioural spec (not code) taken from
 * the reference's utils.c, list.c, option_list.c, tree.c, image.c — cited per function.
 */
#include "y2_host.h"

#include <assert.h>
#include <ctype.h>
#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

/* ---- error conventions (utils.c:195-213): fatal-exit, never an error code ----------- */
void error(const char *s)
{
    perror(s);
    fflush(stderr);
    assert(0);
    exit(-1);
}

void file_error(char *s)
{
    fprintf(stderr, "Couldn't open file: %s\n", s);
    exit(0);
}

void y2_fatal(const char *where, int rc)
{
    fprintf(stderr, "CUDA Error: %s (rc=%d): %s\n", where, rc, y2_last_error());
    fflush(stderr);
    error(where);
}

/* ---- lists (list.c) ------------------------------------------------------------------- */
list *make_list(void)
{
    return (list *)calloc(1, sizeof(list));
}

void list_insert(list *l, void *val)
{
    node *nd = (node *)calloc(1, sizeof(node));
    nd->val = val;
    nd->prev = l->back;
    if (l->back) l->back->next = nd;
    else l->front = nd;
    l->back = nd;
    l->size += 1;
}

void free_list(list *l)
{
    node *n = l->front;
    while (n) {
        node *next = n->next;
        free(n);
        n = next;
    }
    free(l);
}

void free_list_contents(list *l)
{
    for (node *n = l->front; n; n = n->next) free(n->val);
}

void **list_to_array(list *l)
{
    void **a = (void **)calloc(l->size ? l->size : 1, sizeof(void *));
    int i = 0;
    for (node *n = l->front; n; n = n->next) a[i++] = n->val;
    return a;
}

/* ---- text helpers ------------------------------------------------------------------------ */
/* utils.c:263-293: one line without its '\n', NULL at EOF; caller frees */
char *fgetl(FILE *fp)
{
    if (feof(fp)) return 0;
    size_t cap = 512, len = 0;
    char *line = (char *)malloc(cap);
    int ch, got = 0;
    while ((ch = fgetc(fp)) != EOF) {
        got = 1;
        if (ch == '\n') break;
        if (len + 2 > cap) {
            cap *= 2;
            line = (char *)realloc(line, cap);
            if (!line) error("Malloc error");
        }
        line[len++] = (char)ch;
    }
    if (!got) {
        free(line);
        return 0;
    }
    line[len] = '\0';
    return line;
}

/* utils.c:230-241: removes ALL blanks, tabs, CR and LF, not just leading/trailing ones */
void strip(char *s)
{
    char *w = s;
    for (char *r = s; *r; ++r) {
        if (*r == ' ' || *r == '\t' || *r == '\n' || *r == '\r') continue;
        *w++ = *r;
    }
    *w = '\0';
}

/* ---- key=value options (option_list.c) --------------------------------------------------- */
typedef struct {
    char *key;
    char *val;
    int used;
} kvp;

void option_insert(list *l, char *key, char *val)
{
    kvp *p = (kvp *)malloc(sizeof(kvp));
    p->key = key;
    p->val = val;
    p->used = 0;
    list_insert(l, p);
}

/* option_list.c:35-51: splits at the first '='; "key=" (empty value) is rejected */
int read_option(char *s, list *options)
{
    size_t len = strlen(s);
    char *eq = strchr(s, '=');
    if (!eq) return 0;
    if ((size_t)(eq - s) == len - 1) return 0;
    *eq = '\0';
    option_insert(options, s, eq + 1);
    return 1;
}

list *read_data_cfg(char *filename)
{
    FILE *file = fopen(filename, "r");
    if (!file) file_error(filename);
    list *options = make_list();
    char *line;
    int nu = 0;
    while ((line = fgetl(file)) != 0) {
        ++nu;
        strip(line);
        if (line[0] == '\0' || line[0] == '#' || line[0] == ';') {
            free(line);
        } else if (!read_option(line, options)) {
            fprintf(stderr, "Config file error line %d, could parse: %s\n", nu, line);
            free(line);
        }
    }
    fclose(file);
    return options;
}

void option_unused(list *l)
{
    for (node *n = l->front; n; n = n->next) {
        kvp *p = (kvp *)n->val;
        if (!p->used) fprintf(stderr, "Unused field: '%s = %s'\n", p->key, p->val);
    }
}

char *option_find(list *l, char *key)
{
    for (node *n = l->front; n; n = n->next) {
        kvp *p = (kvp *)n->val;
        if (strcmp(p->key, key) == 0) {
            p->used = 1;
            return p->val;
        }
    }
    return 0;
}

char *option_find_str(list *l, char *key, char *def)
{
    char *v = option_find(l, key);
    if (v) return v;
    if (def) fprintf(stderr, "%s: Using default '%s'\n", key, def);
    return def;
}

int option_find_int(list *l, char *key, int def)
{
    char *v = option_find(l, key);
    if (v) return atoi(v);
    fprintf(stderr, "%s: Using default '%d'\n", key, def);
    return def;
}

int option_find_int_quiet(list *l, char *key, int def)
{
    char *v = option_find(l, key);
    return v ? atoi(v) : def;
}

float option_find_float(list *l, char *key, float def)
{
    char *v = option_find(l, key);
    if (v) return (float)atof(v);
    fprintf(stderr, "%s: Using default '%lf'\n", key, def);
    return def;
}

float option_find_float_quiet(list *l, char *key, float def)
{
    char *v = option_find(l, key);
    return v ? (float)atof(v) : def;
}

/* ---- misc readers ------------------------------------------------------------------------- */
/* utils.c:17-33: one integer per line */
int *read_map(char *filename)
{
    FILE *file = fopen(filename, "r");
    if (!file) file_error(filename);
    int n = 0, *map = 0;
    char *str;
    while ((str = fgetl(file))) {
        map = (int *)realloc(map, (size_t)(n + 1) * sizeof(int));
        map[n++] = atoi(str);
        free(str);
    }
    fclose(file);
    return map;
}

/* data.c:474-480 + data.c get_paths: one label per line */
char **get_labels(char *filename)
{
    FILE *file = fopen(filename, "r");
    if (!file) file_error(filename);
    list *lines = make_list();
    char *line;
    while ((line = fgetl(file))) list_insert(lines, line);
    fclose(file);
    char **labels = (char **)list_to_array(lines);
    free_list(lines);
    return labels;
}

/* utils.c:533-545: first maximum wins (strict >), -1 for an empty array */
int max_index(float *a, int n)
{
    if (n <= 0) return -1;
    int best = 0;
    float max = a[0];
    for (int i = 1; i < n; ++i) {
        if (a[i] > max) {
            max = a[i];
            best = i;
        }
    }
    return best;
}

/* utils.c:420-433: avg[j] = (sum_i a[i][j]) / n, accumulated in float */
void mean_arrays(float **a, int n, int els, float *avg)
{
    memset(avg, 0, (size_t)els * sizeof(float));
    for (int j = 0; j < n; ++j)
        for (int i = 0; i < els; ++i) avg[i] += a[j][i];
    for (int i = 0; i < els; ++i) avg[i] /= n;
}

/* utils.c:136-153: "dir/name.ext" -> "name" (caller owns the copy) */
char *basecfg(char *cfgfile)
{
    char *c = cfgfile, *next;
    while ((next = strchr(c, '/'))) c = next + 1;
    c = strdup(c);
    next = strchr(c, '.');
    if (next) *next = 0;
    return c;
}

/* ---- command-line flags (utils.c:62-118): consume the matched argv entries --------------- */
static void del_arg(int argc, char **argv, int index)
{
    for (int i = index; i < argc - 1; ++i) argv[i] = argv[i + 1];
    argv[argc - 1] = 0;
}

int find_arg(int argc, char *argv[], char *arg)
{
    for (int i = 0; i < argc; ++i) {
        if (!argv[i]) continue;
        if (0 == strcmp(argv[i], arg)) {
            del_arg(argc, argv, i);
            return 1;
        }
    }
    return 0;
}

int find_int_arg(int argc, char **argv, char *arg, int def)
{
    for (int i = 0; i < argc - 1; ++i) {
        if (!argv[i]) continue;
        if (0 == strcmp(argv[i], arg)) {
            def = atoi(argv[i + 1]);
            del_arg(argc, argv, i);
            del_arg(argc, argv, i);
            break;
        }
    }
    return def;
}

float find_float_arg(int argc, char **argv, char *arg, float def)
{
    for (int i = 0; i < argc - 1; ++i) {
        if (!argv[i]) continue;
        if (0 == strcmp(argv[i], arg)) {
            def = (float)atof(argv[i + 1]);
            del_arg(argc, argv, i);
            del_arg(argc, argv, i);
            break;
        }
    }
    return def;
}

char *find_char_arg(int argc, char **argv, char *arg, char *def)
{
    for (int i = 0; i < argc - 1; ++i) {
        if (!argv[i]) continue;
        if (0 == strcmp(argv[i], arg)) {
            def = argv[i + 1];
            del_arg(argc, argv, i);
            del_arg(argc, argv, i);
            break;
        }
    }
    return def;
}

/* ---- activations (activations.c:9-62) ----------------------------------------------------- */
static const char *k_act_names[] = {"logistic", "relu",  "relie", "linear",  "ramp",  "tanh", "plse",
                                    "leaky",    "elu",   "loggy", "stair",   "hardtan", "lhtan"};

char *get_activation_string(ACTIVATION a)
{
    if ((int)a >= 0 && (int)a < 13) return (char *)k_act_names[a];
    return "relu";
}

ACTIVATION get_activation(char *s)
{
    for (int i = 0; i < 13; ++i)
        if (strcmp(s, k_act_names[i]) == 0) return (ACTIVATION)i;
    fprintf(stderr, "Couldn't find activation function %s, going with ReLU\n", s);
    return RELU;
}

/* ---- WordTree (tree.c) ------------------------------------------------------------------------ */
/* tree.c:53-103: lines "name parent"; a new softmax group starts whenever the parent changes */
tree *read_tree(char *filename)
{
    FILE *fp = fopen(filename, "r");
    if (!fp) file_error(filename);
    tree *t = (tree *)calloc(1, sizeof(tree));
    char *line;
    int last_parent = -1, group_size = 0, groups = 0, n = 0;
    while ((line = fgetl(fp)) != 0) {
        char *id = (char *)calloc(256, 1);
        int parent = -1;
        sscanf(line, "%255s %d", id, &parent);
        t->parent = (int *)realloc(t->parent, (size_t)(n + 1) * sizeof(int));
        t->parent[n] = parent;
        t->name = (char **)realloc(t->name, (size_t)(n + 1) * sizeof(char *));
        t->name[n] = id;
        if (parent != last_parent) {
            ++groups;
            t->group_offset = (int *)realloc(t->group_offset, (size_t)groups * sizeof(int));
            t->group_offset[groups - 1] = n - group_size;
            t->group_size = (int *)realloc(t->group_size, (size_t)groups * sizeof(int));
            t->group_size[groups - 1] = group_size;
            group_size = 0;
            last_parent = parent;
        }
        t->group = (int *)realloc(t->group, (size_t)(n + 1) * sizeof(int));
        t->group[n] = groups;
        ++n;
        ++group_size;
        free(line);
    }
    ++groups;
    t->group_offset = (int *)realloc(t->group_offset, (size_t)groups * sizeof(int));
    t->group_offset[groups - 1] = n - group_size;
    t->group_size = (int *)realloc(t->group_size, (size_t)groups * sizeof(int));
    t->group_size[groups - 1] = group_size;
    t->n = n;
    t->groups = groups;
    t->leaf = (int *)calloc(n ? n : 1, sizeof(int));
    for (int i = 0; i < n; ++i) t->leaf[i] = 1;
    for (int i = 0; i < n; ++i)
        if (t->parent[i] >= 0) t->leaf[t->parent[i]] = 0;
    fclose(fp);
    return t;
}

/* tree.c:37-51 (host helper; the device path is region_boxes_tree_kernel) */
void hierarchy_predictions(float *predictions, int n, tree *hier, int only_leaves)
{
    for (int j = 0; j < n; ++j) {
        int parent = hier->parent[j];
        if (parent >= 0) predictions[j] *= predictions[parent];
    }
    if (only_leaves)
        for (int j = 0; j < n; ++j)
            if (!hier->leaf[j]) predictions[j] = 0;
}

/* tree.c:26-35 */
float get_hierarchy_probability(float *x, tree *hier, int c)
{
    float p = 1;
    while (c >= 0) {
        p = p * x[c];
        c = hier->parent[c];
    }
    return p;
}

/* ---- images ----------------------------------------------------------------------------------- */
image make_image(int w, int h, int c)
{
    image out;
    out.w = w;
    out.h = h;
    out.c = c;
    out.data = (float *)calloc((size_t)h * w * c, sizeof(float));
    return out;
}

void free_image(image m)
{
    if (m.data) free(m.data);
}

static inline float px(image m, int x, int y, int c)
{
    return m.data[((size_t)c * m.h + y) * m.w + x];
}

/* image.c:1950-1993: two-pass bilinear, first along x into a (w x im.h) image, then along y;
 * scales (in-1)/(out-1); the last column/row copies the source edge; the y pass accumulates
 * (1-dy)*row[iy] first and adds dy*row[iy+1] afterwards. */
image resize_image(image im, int w, int h)
{
    image resized = make_image(w, h, im.c);
    image part = make_image(w, im.h, im.c);
    float w_scale = (float)(im.w - 1) / (w - 1);
    float h_scale = (float)(im.h - 1) / (h - 1);
    for (int k = 0; k < im.c; ++k) {
        for (int r = 0; r < im.h; ++r) {
            for (int c = 0; c < w; ++c) {
                float val;
                if (c == w - 1 || im.w == 1) {
                    val = px(im, im.w - 1, r, k);
                } else {
                    float sx = c * w_scale;
                    int ix = (int)sx;
                    float dx = sx - ix;
                    val = (1 - dx) * px(im, ix, r, k) + dx * px(im, ix + 1, r, k);
                }
                part.data[((size_t)k * part.h + r) * part.w + c] = val;
            }
        }
    }
    for (int k = 0; k < im.c; ++k) {
        for (int r = 0; r < h; ++r) {
            float sy = r * h_scale;
            int iy = (int)sy;
            float dy = sy - iy;
            for (int c = 0; c < w; ++c) {
                float val = (1 - dy) * px(part, c, iy, k);
                resized.data[((size_t)k * h + r) * w + c] = val;
            }
            if (r == h - 1 || im.h == 1) continue;
            for (int c = 0; c < w; ++c) {
                float val = dy * px(part, c, iy + 1, k);
                resized.data[((size_t)k * h + r) * w + c] += val;
            }
        }
    }
    free_image(part);
    return resized;
}

/* ---- classifier front end (classifier.c:676-730 predict_classifier): letterbox + top-k ---------------- */

/* image.c:1601-1605 */
void fill_image(image m, float s)
{
    const size_t n = (size_t)m.h * m.w * m.c;
    for (size_t i = 0; i < n; ++i) m.data[i] = s;
}

/* image.c:1087-1098: paste `source` into `dest` with its top-left corner at (dx, dy); pixels that fall
 * outside dest are dropped (the reference asserts) */
void embed_image(image source, image dest, int dx, int dy)
{
    for (int k = 0; k < source.c && k < dest.c; ++k)
        for (int y = 0; y < source.h; ++y) {
            const int ty = dy + y;
            if (ty < 0 || ty >= dest.h) continue;
            for (int x = 0; x < source.w; ++x) {
                const int tx = dx + x;
                if (tx < 0 || tx >= dest.w) continue;
                dest.data[((size_t)k * dest.h + ty) * dest.w + tx] = px(source, x, y, k);
            }
        }
}

/* image.c:1624-1644: scale to fit inside w x h keeping the aspect ratio (y2_letterbox_geometry), centre on a
 * 0.5-grey canvas */
image letterbox_image(image im, int w, int h)
{
    int new_w, new_h, dx, dy;
    y2_letterbox_geometry(im.w, im.h, w, h, &new_w, &new_h, &dx, &dy);
    image resized = resize_image(im, new_w, new_h);
    image boxed = make_image(w, h, im.c);
    fill_image(boxed, .5f);
    embed_image(resized, boxed, dx, dy);
    free_image(resized);
    return boxed;
}

/* utils.c:179-193: indices of the k largest entries, descending; among equal values the one met first
 * stays ahead (the comparison that displaces an entry is a strict >) */
void top_k(float *a, int n, int k, int *index)
{
    for (int j = 0; j < k; ++j) index[j] = -1;
    for (int i = 0; i < n; ++i) {
        int curr = i;
        for (int j = 0; j < k; ++j) {
            if (index[j] < 0 || a[curr] > a[index[j]]) {
                const int displaced = index[j];
                index[j] = curr;
                curr = displaced;
            }
            if (curr < 0) break; /* nothing left to push down */
        }
    }
}
