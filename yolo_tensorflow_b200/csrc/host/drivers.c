/*
 * drivers.c — the host helpers that examples/detector.c, examples/yolo.c and examples/darknet.c call AROUND the accelerated
 * path (SURVEY.md §8b "also needed for the drivers to link/run unchanged"): the option list of `.data` files, command-line
 * argument scanning, label lists, the glyph alphabet, box/label drawing and the PNG writer of the CPU build.  Plain host C
 * re-statements of the reference's behaviour (list.c, option_list.c:7-140, utils.c:89-199,302-368, data.c:12-23,618-624,
 * image.c:17-26,92-240,239-316,696-720); nothing here touches the device.
 *
 * Differences, on purpose: images are read by this library's load_image_color (binary PPM/PGM; the reference decodes through
 * the vendored stb_image), so load_alphabet() expects data/labels/<char>_<size>.png to hold PNM data when used with this
 * library alone; save_image() writes a valid PNG with stored (uncompressed) deflate blocks instead of stb's compressor — same
 * pixels, larger file; instance-mask overlays of draw_detections (coords > 4) are not drawn.
 */
#include "darknet.h"
#include <math.h>
#include <stdint.h>

/* ---- list.c ------------------------------------------------------------------------------------------------------- */
list *make_list(void)
{
    list *l = calloc(1, sizeof(list));
    return l;
}

void list_insert(list *l, void *val)
{
    node *n = malloc(sizeof(node));
    n->val = val; n->next = NULL; n->prev = l->back;
    if (l->back) l->back->next = n; else l->front = n;
    l->back = n;
    l->size += 1;
}

void free_list(list *l)
{
    for (node *n = l->front; n;) { node *next = n->next; free(n); n = next; }
    free(l);
}

void **list_to_array(list *l)
{
    void **a = calloc(l->size > 0 ? l->size : 1, sizeof(void *));
    int k = 0;
    for (node *n = l->front; n; n = n->next) a[k++] = n->val;
    return a;
}

/* ---- utils.c: lines, blanks, arguments ------------------------------------------------------------------------------ */
char *fgetl(FILE *fp)                              /* utils.c:335-368: one line without its '\n', NULL at end of file */
{
    char *line = NULL;
    size_t cap = 0;
    ssize_t len = getline(&line, &cap, fp);
    if (len < 0) { free(line); return NULL; }
    if (len > 0 && line[len - 1] == '\n') line[len - 1] = 0;
    return line;
}

void strip(char *s)                                /* utils.c:302-313: drops ' ', '\t', '\n' everywhere */
{
    char *w = s;
    for (char *r = s; *r; ++r) if (*r != ' ' && *r != '\t' && *r != '\n') *w++ = *r;
    *w = 0;
}

static void drop_arg(int argc, char **argv, int index)          /* utils.c:109-118 */
{
    for (int i = index; i < argc - 1; ++i) argv[i] = argv[i + 1];
    argv[argc - 1] = NULL;
}

int find_arg(int argc, char *argv[], char *arg)
{
    for (int i = 0; i < argc; ++i)
        if (argv[i] && strcmp(argv[i], arg) == 0) { drop_arg(argc, argv, i); return 1; }
    return 0;
}

static int find_valued(int argc, char **argv, const char *arg)   /* index of the value of `-flag value`, both removed afterwards */
{
    for (int i = 0; i < argc - 1; ++i)
        if (argv[i] && strcmp(argv[i], arg) == 0) return i + 1;
    return -1;
}

int find_int_arg(int argc, char **argv, char *arg, int def)
{
    int v = find_valued(argc, argv, arg);
    if (v < 0) return def;
    def = atoi(argv[v]);
    drop_arg(argc, argv, v - 1); drop_arg(argc, argv, v - 1);
    return def;
}

float find_float_arg(int argc, char **argv, char *arg, float def)
{
    int v = find_valued(argc, argv, arg);
    if (v < 0) return def;
    def = atof(argv[v]);
    drop_arg(argc, argv, v - 1); drop_arg(argc, argv, v - 1);
    return def;
}

char *find_char_arg(int argc, char **argv, char *arg, char *def)
{
    int v = find_valued(argc, argv, arg);
    if (v < 0) return def;
    def = argv[v];
    drop_arg(argc, argv, v - 1); drop_arg(argc, argv, v - 1);
    return def;
}

char *basecfg(char *cfgfile)                       /* utils.c:179-191: file name without directories and extension */
{
    char *slash = strrchr(cfgfile, '/');
    char *c = strdup(slash ? slash + 1 : cfgfile);
    char *dot = strchr(c, '.');
    if (dot) *dot = 0;
    return c;
}

/* utils.c top_k: the k largest entries of a[n], descending, by insertion with a strict `>` (what predict_classifier
 * and classify() rank with).  An entry displaced from slot j moves on only past strictly smaller entries, so equal values do not
 * always keep index order (e.g. {5, 5, 3} then 6 gives 6, a[1], a[0]); the device top-k reproduces exactly this order. */
void top_k(float *a, int n, int k, int *index)
{
    for (int j = 0; j < k; ++j) index[j] = -1;
    for (int i = 0; i < n; ++i) {
        int curr = i;
        for (int j = 0; j < k; ++j) {
            if (index[j] < 0 || a[curr] > a[index[j]]) {
                int swap = curr;
                curr = index[j];
                index[j] = swap;
            }
        }
    }
}

/* ---- option_list.c ------------------------------------------------------------------------------------------------------ */
typedef struct { char *key, *val; int used; } kvp;                 /* option_list.h:6-10 */

list *read_data_cfg(char *filename)
{
    FILE *fp = fopen(filename, "r");
    if (!fp) { fprintf(stderr, "Couldn't open file: %s\n", filename); exit(0); }     /* file_error, utils.c:281-285 */
    list *options = make_list();
    char *line;
    int nu = 0;
    while ((line = fgetl(fp)) != NULL) {
        ++nu;
        strip(line);
        if (line[0] == 0 || line[0] == '#' || line[0] == ';') { free(line); continue; }
        char *eq = strchr(line, '=');
        /* read_option (:52-68): no '=' or '=' as the last character is an error line */
        if (!eq || eq[1] == 0) {
            fprintf(stderr, "Config file error line %d, could parse: %s\n", nu, line);
            free(line);
            continue;
        }
        *eq = 0;
        kvp *p = malloc(sizeof(kvp));
        p->key = line; p->val = eq + 1; p->used = 0;
        list_insert(options, p);
    }
    fclose(fp);
    return options;
}

char *option_find(list *l, char *key)
{
    for (node *n = l->front; n; n = n->next) {
        kvp *p = n->val;
        if (strcmp(p->key, key) == 0) { p->used = 1; return p->val; }
    }
    return NULL;
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
    if (v) return atof(v);
    fprintf(stderr, "%s: Using default '%lf'\n", key, def);
    return def;
}

float option_find_float_quiet(list *l, char *key, float def)
{
    char *v = option_find(l, key);
    return v ? atof(v) : def;
}

void option_unused(list *l)
{
    for (node *n = l->front; n; n = n->next) {
        kvp *p = n->val;
        if (!p->used) fprintf(stderr, "Unused field: '%s = %s'\n", p->key, p->val);
    }
}

/* ---- data.c: path / label lists -------------------------------------------------------------------------------------------- */
list *get_paths(char *filename)
{
    FILE *fp = fopen(filename, "r");
    if (!fp) { fprintf(stderr, "Couldn't open file: %s\n", filename); exit(0); }
    list *lines = make_list();
    char *path;
    while ((path = fgetl(fp)) != NULL) list_insert(lines, path);
    fclose(fp);
    return lines;
}

char **get_labels(char *filename)
{
    list *l = get_paths(filename);
    char **labels = (char **)list_to_array(l);
    free_list(l);
    return labels;
}

int *read_map(char *filename)                      /* utils.c:62-77: one class index per line (coco9k.map, inet9k.map) */
{
    FILE *fp = fopen(filename, "r");
    if (!fp) { fprintf(stderr, "Couldn't open file: %s\n", filename); exit(0); }
    int n = 0, *map = NULL;
    char *str;
    while ((str = fgetl(fp)) != NULL) {
        map = realloc(map, (size_t)(n + 1) * sizeof(int));
        map[n++] = atoi(str);
        free(str);
    }
    fclose(fp);
    return map;
}

/* ---- tree.c: the WordTree of YOLO9000 (`tree=` of a [region] layer, SURVEY §8f-4) ---------------------------------------- */
tree *read_tree(char *filename)
{
    /* tree.c:83-139: one "<name> <parent index>" line per class; consecutive classes with the same parent form a group (the
     * unit the softmax runs over); child[i] = group of i's children, or -1 */
    FILE *fp = fopen(filename, "r");
    if (!fp) { fprintf(stderr, "Couldn't open file: %s\n", filename); exit(0); }
    tree *t = calloc(1, sizeof(tree));
    int n = 0, groups = 0, group_size = 0, last_parent = -1;
    char *line;
    while ((line = fgetl(fp)) != NULL) {
        char *id = calloc(256, sizeof(char));
        int parent = -1;
        sscanf(line, "%255s %d", id, &parent);
        free(line);
        t->parent = realloc(t->parent, (size_t)(n + 1) * sizeof(int));
        t->child  = realloc(t->child,  (size_t)(n + 1) * sizeof(int));
        t->name   = realloc(t->name,   (size_t)(n + 1) * sizeof(char *));
        t->group  = realloc(t->group,  (size_t)(n + 1) * sizeof(int));
        t->parent[n] = parent; t->child[n] = -1; t->name[n] = id;
        if (parent != last_parent) {                     /* a new group starts: close the previous one */
            ++groups;
            t->group_offset = realloc(t->group_offset, (size_t)groups * sizeof(int));
            t->group_size   = realloc(t->group_size,   (size_t)groups * sizeof(int));
            t->group_offset[groups - 1] = n - group_size;
            t->group_size[groups - 1] = group_size;
            group_size = 0;
            last_parent = parent;
        }
        t->group[n] = groups;
        if (parent >= 0) t->child[parent] = groups;
        ++n; ++group_size;
    }
    fclose(fp);
    ++groups;
    t->group_offset = realloc(t->group_offset, (size_t)groups * sizeof(int));
    t->group_size   = realloc(t->group_size,   (size_t)groups * sizeof(int));
    t->group_offset[groups - 1] = n - group_size;
    t->group_size[groups - 1] = group_size;
    t->n = n; t->groups = groups;
    t->leaf = calloc(n > 0 ? n : 1, sizeof(int));
    for (int i = 0; i < n; ++i) t->leaf[i] = 1;
    for (int i = 0; i < n; ++i) if (t->parent[i] >= 0) t->leaf[t->parent[i]] = 0;
    return t;
}

void hierarchy_predictions(float *predictions, int n, tree *hier, int only_leaves, int stride)
{
    /* tree.c:37-51, host version for drivers; the engine runs the same recurrence on the device (dev/heads.cu) */
    for (int j = 0; j < n; ++j) {
        int parent = hier->parent[j];
        if (parent >= 0) predictions[j * stride] *= predictions[parent * stride];
    }
    if (only_leaves) for (int j = 0; j < n; ++j) if (!hier->leaf[j]) predictions[j * stride] = 0;
}

int hierarchy_top_prediction(float *predictions, tree *hier, float thresh, int stride)
{
    /* tree.c:53-81: walk down from the root group, always into the most probable child, while the path stays over thresh */
    float p = 1;
    int group = 0;
    for (;;) {
        float best = 0;
        int best_i = 0;
        for (int i = 0; i < hier->group_size[group]; ++i) {
            int index = i + hier->group_offset[group];
            float val = predictions[index * stride];
            if (val > best) { best_i = index; best = val; }
        }
        if (p * best > thresh) {
            p = p * best;
            group = hier->child[best_i];
            if (hier->child[best_i] < 0) return best_i;
        } else if (group == 0) {
            return best_i;
        } else {
            return hier->parent[hier->group_offset[group]];
        }
    }
}

/* ---- image.c: drawing --------------------------------------------------------------------------------------------------------- */
static float px_get(image m, int x, int y, int c) { return m.data[((size_t)c * m.h + y) * m.w + x]; }
static float px_get_or_zero(image m, int x, int y, int c)
{
    if (x < 0 || x >= m.w || y < 0 || y >= m.h || c < 0 || c >= m.c) return 0;
    return px_get(m, x, y, c);
}
static void px_set(image m, int x, int y, int c, float v)
{
    if (x < 0 || y < 0 || c < 0 || x >= m.w || y >= m.h || c >= m.c) return;
    m.data[((size_t)c * m.h + y) * m.w + x] = v;
}

image copy_image(image p)
{
    image c = p;
    c.data = calloc((size_t)p.w * p.h * p.c > 0 ? (size_t)p.w * p.h * p.c : 1, sizeof(float));
    memcpy(c.data, p.data, (size_t)p.w * p.h * p.c * sizeof(float));
    return c;
}

float get_color(int c, int x, int max)             /* image.c:15-26: six-colour wheel, linear between neighbours */
{
    static const float wheel[6][3] = {{1, 0, 1}, {0, 0, 1}, {0, 1, 1}, {0, 1, 0}, {1, 1, 0}, {1, 0, 0}};
    float ratio = ((float)x / max) * 5;
    int i = floor(ratio), j = ceil(ratio);
    ratio -= i;
    return (1 - ratio) * wheel[i][c] + ratio * wheel[j][c];
}

void draw_box(image a, int x1, int y1, int x2, int y2, float r, float g, float b)
{
    const float rgb[3] = {r, g, b};
    const size_t plane = (size_t)a.w * a.h;
    x1 = x1 < 0 ? 0 : (x1 >= a.w ? a.w - 1 : x1);
    x2 = x2 < 0 ? 0 : (x2 >= a.w ? a.w - 1 : x2);
    y1 = y1 < 0 ? 0 : (y1 >= a.h ? a.h - 1 : y1);
    y2 = y2 < 0 ? 0 : (y2 >= a.h ? a.h - 1 : y2);
    for (int k = 0; k < 3; ++k) {
        float *p = a.data + k * plane;
        for (int i = x1; i <= x2; ++i) { p[i + (size_t)y1 * a.w] = rgb[k]; p[i + (size_t)y2 * a.w] = rgb[k]; }
        for (int i = y1; i <= y2; ++i) { p[x1 + (size_t)i * a.w] = rgb[k]; p[x2 + (size_t)i * a.w] = rgb[k]; }
    }
}

void draw_box_width(image a, int x1, int y1, int x2, int y2, int w, float r, float g, float b)
{
    for (int i = 0; i < w; ++i) draw_box(a, x1 + i, y1 + i, x2 - i, y2 - i, r, g, b);
}

/* b appended to the right of a with a horizontal gap of dx (may be negative): white canvas, a copied, b MULTIPLIED in
 * (tile_images + composite_image, image.c:92-130) */
static image append_glyph(image a, image b, int dx)
{
    if (a.w == 0) return copy_image(b);
    image c = make_image(a.w + b.w + dx, a.h > b.h ? a.h : b.h, a.c > b.c ? a.c : b.c);
    for (size_t i = 0; i < (size_t)c.w * c.h * c.c; ++i) c.data[i] = 1;
    for (int k = 0; k < a.c; ++k)
        for (int y = 0; y < a.h; ++y)
            for (int x = 0; x < a.w; ++x) px_set(c, x, y, k, px_get(a, x, y, k));
    for (int k = 0; k < b.c; ++k)
        for (int y = 0; y < b.h; ++y)
            for (int x = 0; x < b.w; ++x) px_set(c, a.w + dx + x, y, k, px_get(b, x, y, k) * px_get_or_zero(c, a.w + dx + x, y, k));
    return c;
}

image get_label(image **characters, char *string, int size)      /* image.c:132-147 */
{
    size = size / 10;
    if (size > 7) size = 7;
    image label = {0, 0, 0, NULL};
    for (; *string; ++string) {
        image glyph = characters[size][(int)*string];
        image next = append_glyph(label, glyph, -size - 1 + (size + 1) / 2);
        free_image(label);
        label = next;
    }
    const int border = label.h * .25;                              /* white frame of a quarter of the glyph height */
    image framed = make_image(label.w + 2 * border, label.h + 2 * border, label.c);
    for (int k = 0; k < framed.c; ++k)
        for (int y = 0; y < framed.h; ++y)
            for (int x = 0; x < framed.w; ++x) {
                const int sx = x - border, sy = y - border;
                const int outside = sx < 0 || sx >= label.w || sy < 0 || sy >= label.h;
                px_set(framed, x, y, k, outside ? 1 : px_get(label, sx, sy, k));
            }
    free_image(label);
    return framed;
}

void draw_label(image a, int r, int c, image label, const float *rgb)      /* image.c:149-164 */
{
    if (r - label.h >= 0) r -= label.h;
    for (int j = 0; j < label.h && j + r < a.h; ++j)
        for (int i = 0; i < label.w && i + c < a.w; ++i)
            for (int k = 0; k < label.c; ++k) px_set(a, i + c, j + r, k, rgb[k] * px_get(label, i, j, k));
}

image **load_alphabet(void)                        /* image.c:223-237: 8 sizes x printable ASCII from data/labels/ */
{
    const int nsize = 8;
    image **alphabets = calloc(nsize, sizeof(image *));
    for (int j = 0; j < nsize; ++j) {
        alphabets[j] = calloc(128, sizeof(image));
        for (int i = 32; i < 127; ++i) {
            char path[256];
            snprintf(path, sizeof path, "data/labels/%d_%d.png", i, j);
            alphabets[j][i] = load_image_color(path, 0, 0);
        }
    }
    return alphabets;
}

void draw_detections(image im, detection *dets, int num, float thresh, char **names, image **alphabet, int classes)
{
    /* image.c:239-316: one stdout line per (detection, class) over the threshold, one box + label per detection */
    for (int i = 0; i < num; ++i) {
        char labelstr[4096] = {0};
        int first = -1;
        for (int j = 0; j < classes; ++j) {
            if (!(dets[i].prob[j] > thresh)) continue;
            if (first >= 0) strncat(labelstr, ", ", sizeof labelstr - strlen(labelstr) - 1);
            else first = j;
            strncat(labelstr, names[j], sizeof labelstr - strlen(labelstr) - 1);
            printf("%s: %.0f%%\n", names[j], dets[i].prob[j] * 100);
        }
        if (first < 0) continue;
        const int width = im.h * .006;
        const int offset = first * 123457 % classes;
        const float rgb[3] = {get_color(2, offset, classes), get_color(1, offset, classes), get_color(0, offset, classes)};
        const box b = dets[i].bbox;
        int left = (b.x - b.w / 2.) * im.w, right = (b.x + b.w / 2.) * im.w;
        int top = (b.y - b.h / 2.) * im.h, bot = (b.y + b.h / 2.) * im.h;
        if (left < 0) left = 0;
        if (right > im.w - 1) right = im.w - 1;
        if (top < 0) top = 0;
        if (bot > im.h - 1) bot = im.h - 1;
        draw_box_width(im, left, top, right, bot, width, rgb[0], rgb[1], rgb[2]);
        if (alphabet) {
            image label = get_label(alphabet, labelstr, (im.h * .03));
            draw_label(im, top + width, left, label, rgb);
            free_image(label);
        }
    }
}

/* ---- PNG writer (image.c:696-720 writes <name>.png through stb_image_write; here: stored deflate blocks) ------------------ */
static uint32_t crc32_of(const unsigned char *p, size_t n, uint32_t crc)
{
    static uint32_t table[256];
    static int ready = 0;
    if (!ready) {
        for (uint32_t i = 0; i < 256; ++i) { uint32_t c = i; for (int k = 0; k < 8; ++k) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1; table[i] = c; }
        ready = 1;
    }
    crc = ~crc;
    for (size_t i = 0; i < n; ++i) crc = table[(crc ^ p[i]) & 0xFF] ^ (crc >> 8);
    return ~crc;
}

static void put_be32(unsigned char *p, uint32_t v) { p[0] = v >> 24; p[1] = v >> 16; p[2] = v >> 8; p[3] = v; }

static void png_chunk(FILE *fp, const char *type, const unsigned char *data, uint32_t len)
{
    unsigned char hdr[8], tail[4];
    put_be32(hdr, len); memcpy(hdr + 4, type, 4);
    uint32_t crc = crc32_of(hdr + 4, 4, 0);
    if (len) crc = crc32_of(data, len, crc);
    put_be32(tail, crc);
    fwrite(hdr, 1, 8, fp);
    if (len) fwrite(data, 1, len, fp);
    fwrite(tail, 1, 4, fp);
}

void save_image_png(image im, const char *name)
{
    char path[256];
    snprintf(path, sizeof path, "%s.png", name);
    if (im.c != 1 && im.c != 3 && im.c != 4) { fprintf(stderr, "Failed to write image %s\n", path); return; }
    FILE *fp = fopen(path, "wb");
    if (!fp) { fprintf(stderr, "Failed to write image %s\n", path); return; }
    const size_t row = (size_t)im.w * im.c + 1, raw_len = row * im.h, plane = (size_t)im.w * im.h;
    unsigned char *raw = malloc(raw_len ? raw_len : 1);
    for (int y = 0; y < im.h; ++y) {
        raw[y * row] = 0;                                          /* filter type 0 */
        for (int x = 0; x < im.w; ++x)
            for (int k = 0; k < im.c; ++k)
                raw[y * row + 1 + (size_t)x * im.c + k] = (unsigned char)(255 * im.data[(size_t)y * im.w + x + k * plane]);
    }
    /* zlib stream: header, stored blocks of at most 65535 bytes, adler32 */
    const size_t blocks = raw_len / 65535 + 1;
    unsigned char *z = malloc(2 + raw_len + 5 * blocks + 4);
    size_t o = 0;
    z[o++] = 0x78; z[o++] = 0x01;
    uint32_t s1 = 1, s2 = 0;
    for (size_t off = 0, b = 0; b < blocks; ++b) {
        const size_t n = raw_len - off < 65535 ? raw_len - off : 65535;
        z[o++] = (b == blocks - 1) ? 1 : 0;
        z[o++] = n & 0xFF; z[o++] = n >> 8; z[o++] = ~n & 0xFF; z[o++] = (~n >> 8) & 0xFF;
        memcpy(z + o, raw + off, n);
        for (size_t i = 0; i < n; ++i) { s1 = (s1 + raw[off + i]) % 65521; s2 = (s2 + s1) % 65521; }
        o += n; off += n;
    }
    put_be32(z + o, (s2 << 16) | s1); o += 4;
    static const unsigned char sig[8] = {0x89, 'P', 'N', 'G', '\r', '\n', 0x1A, '\n'};
    unsigned char ihdr[13];
    put_be32(ihdr, im.w); put_be32(ihdr + 4, im.h);
    ihdr[8] = 8; ihdr[9] = im.c == 1 ? 0 : (im.c == 3 ? 2 : 6); ihdr[10] = ihdr[11] = ihdr[12] = 0;
    fwrite(sig, 1, 8, fp);
    png_chunk(fp, "IHDR", ihdr, 13);
    png_chunk(fp, "IDAT", z, (uint32_t)o);
    png_chunk(fp, "IEND", NULL, 0);
    fclose(fp);
    free(raw); free(z);
}

void save_image(image im, const char *name) { save_image_png(im, name); }   /* image.c:713-720 with OPENCV undefined */
