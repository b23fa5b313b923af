/* The two root rules of the engine's search for the CPU oracle: forced
 * playouts (Wu 2019, "Accelerating Self-Play Learning in Go", section 3.2;
 * az_engine_set_forced_playouts) and Dirichlet root noise (mcts.py:126-131).
 * TEST INFRASTRUCTURE ONLY.
 *
 * select_batch below is omcts_select_batch (azalea_oracle.c, mcts.py:46-76)
 * with both rules added at the root:
 *  - root noise: with noise != NULL and noise_scale != 0, descent i of the
 *    call scores the root's children with P'[j] = (float)((1 - eps) * (double)
 *    P[j] + eps * (double)noise[i][j]), mixed in double (k_select), where the
 *    noise array is [batch][k_root].  The noise vectors are given, not drawn:
 *    the device's own draws (Engine.noise_sample) make the search comparable
 *    bit for bit;
 *  - forced playouts: with forced_k != 0 a root child with 0 < N <
 *    sqrtf((forced_k * P) * sum N) scores +inf, so np.argmax takes the lowest
 *    such ordinal.  P is the stored prior, not the noised one; N and sum N
 *    include the batch's virtual losses.
 * float32 otherwise, one rounding per operation.  With forced_k = 0 and no
 * noise every entry point is bit for bit the oracle's own (tested).
 * Everything else goes through the oracle's exported functions: this file is
 * linked against libazalea_oracle.so and works on its trees. */
#include "azalea_oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>

static void apply_virtual_loss(otree *t, int32_t node, float amount)
{
    /* mcts.py:79-92: leaf .. child-of-root; the root is not touched */
    while (node != t->root_id) {
        t->num_visits[node] += amount;
        t->total_value[node] += amount;
        node = t->parent[node];
    }
}

static void leaf_state(const ohex *g, oleaves *out, int slot)
{
    /* GameState at the leaf (hex.py:55-60) turned into the network's view
     * (mcts.py:176-181) */
    int32_t legal[19 * 19];
    int nn = g->n * g->n;
    int k = ohex_legal_moves(g, legal);
    out->color[slot] = g->color - 1;
    out->result[slot] = ohex_result(g);
    out->num_moves[slot] = k;
    if (g->color - 1 == 1) {
        ohex_flip_board(g->board, g->n, out->board_view[slot]);
        ohex_flip_moves(legal, k, g->n, out->moves_view[slot]);
    } else {
        memcpy(out->board_view[slot], g->board, sizeof(int32_t) * nn);
        memcpy(out->moves_view[slot], legal, sizeof(int32_t) * k);
    }
}

/* How the root noise is mixed into the prior: OMIX_F64 is the engine's rule.
 * The float32 variants exist only so that a test can ask whether a search
 * would notice a kernel that mixed in float32. */
enum { OMIX_F64 = 0, OMIX_F32 = 1, OMIX_F32_FMA = 2 };

static float mix_prior(float p, float eta, double eps, int mix)
{
    if (mix == OMIX_F32)
        return (1.0f - (float)eps) * p + (float)eps * eta;
    if (mix == OMIX_F32_FMA)
        return fmaf((float)eps, eta, (1.0f - (float)eps) * p);
    return (float)((1.0 - eps) * (double)p + eps * (double)eta);
}

static int select_batch(otree *t, const ohex *game, int batch_size, float coef,
                        float forced_k, double noise_scale, const float *noise,
                        int mix, oleaves *out)
{
    int32_t leaf_nodes[OMAX_BATCH];
    static __thread ohex leaf_games[OMAX_BATCH];
    float nv[19 * 19], ntv[19 * 19], pr[19 * 19], pm[19 * 19], score[19 * 19];
    const int32_t k_root = t->num_children[t->root_id];
    if (batch_size > OMAX_BATCH || k_root <= 0)
        return -1;
    if (noise_scale == 0.0)
        noise = NULL;
    out->sum_children = 0;
    out->sum_depth = 0;
    for (int i = 0; i < batch_size; i++) {
        ohex g = *game;
        int32_t node = t->root_id;
        while (t->num_children[node] > 0) {
            int32_t k = t->num_children[node], fc = t->first_child[node];
            int32_t legal[19 * 19];
            int best = 0;
            for (int j = 0; j < k; j++) {
                nv[j] = t->num_visits[fc + j];
                ntv[j] = -t->total_value[fc + j];
                pr[j] = t->prior_prob[fc + j];
            }
            if (noise && node == t->root_id) {
                const float *eta = noise + (size_t)i * k_root;
                for (int j = 0; j < k; j++)
                    pm[j] = mix_prior(pr[j], eta[j], noise_scale, mix);
                omcts_score_actions(nv, ntv, pm, k, coef, score);
            } else {
                omcts_score_actions(nv, ntv, pr, k, coef, score);
            }
            if (forced_k != 0.0f && node == t->root_id) {
                double s = 0;           /* sum of small integers: exact */
                for (int j = 0; j < k; j++)
                    s += nv[j];
                for (int j = 0; j < k; j++) {
                    float nf = sqrtf((forced_k * pr[j]) * (float)s);
                    if (nv[j] > 0.0f && nv[j] < nf)
                        score[j] = INFINITY;
                }
            }
            for (int j = 1; j < k; j++)  /* np.argmax: first maximum */
                if (score[j] > score[best])
                    best = j;
            if (ohex_legal_moves(&g, legal) != k)
                return -2;
            ohex_step(&g, legal[best]);
            node = fc + best;
            out->sum_children += k;
            out->sum_depth += 1;
        }
        apply_virtual_loss(t, node, 1.0f);
        leaf_nodes[i] = node;
        leaf_games[i] = g;
    }
    for (int i = 0; i < batch_size; i++)
        apply_virtual_loss(t, leaf_nodes[i], -1.0f);
    /* deduplicate_leaves, mcts.py:139-152 */
    out->count = 0;
    for (int i = 0; i < batch_size; i++) {
        int seen = 0;
        for (int q = 0; q < out->count; q++)
            if (out->node[q] == leaf_nodes[i])
                seen = 1;
        if (seen)
            continue;
        out->node[out->count] = leaf_nodes[i];
        leaf_state(&leaf_games[i], out, out->count);
        out->count++;
    }
    return out->count;
}

int omcts_select_batch_forced(otree *t, const ohex *game, int batch_size,
                              float coef, float forced_k, oleaves *out)
{
    return select_batch(t, game, batch_size, coef, forced_k, 0.0, NULL, OMIX_F64, out);
}

/* Both root rules; noise is [batch_size][k_root] (may be NULL). */
int omcts_select_batch_noise(otree *t, const ohex *game, int batch_size,
                             float coef, float forced_k, double noise_scale,
                             const float *noise, int mix, oleaves *out)
{
    return select_batch(t, game, batch_size, coef, forced_k, noise_scale, noise, mix, out);
}

static void eval_stub(const oleaves *lv, int n, int mode, float *value,
                      float *prior, int stride)
{
    for (int i = 0; i < lv->count; i++) {
        if (lv->result[i] != 0) {
            value[i] = -1.0f;
            continue;
        }
        ostub_eval(mode, lv->board_view[i], n, lv->moves_view[i],
                   lv->num_moves[i], &value[i], prior + (size_t)i * stride);
    }
}

/* omcts_sample_paths_stub (mcts.py:258-293) with both root rules: the
 * call's b-th select uses noise rows b * batch_size .. b * batch_size +
 * batch_size - 1 of noise[num_batches * batch_size][k_root].  Returns -1 on
 * SearchTreeFull. */
static int sample_paths_stub(otree *t, const ohex *game, int num_simulations,
                             int batch_size, float coef, float forced_k,
                             double noise_scale, const float *noise, int mix,
                             int stub_mode, float *search_value)
{
    int num_batches = num_simulations / batch_size + 1;
    int stride = 19 * 19;
    float value[OMAX_BATCH];
    float sv_total = 0;
    int rc = 0;
    oleaves *lv = (oleaves *)malloc(sizeof(oleaves));
    float *prior = (float *)malloc(sizeof(float) * OMAX_BATCH * 19 * 19);
    if (!lv || !prior) {
        rc = -1;
        goto done;
    }
    if (t->num_children[t->root_id] < 0) {
        omcts_root_leaf(t, game, lv);
        eval_stub(lv, game->n, stub_mode, value, prior, stride);
        if (omcts_expand_root(t, lv, prior)) {
            rc = -1;
            goto done;
        }
    }
    for (int b = 0; b < num_batches; b++) {
        float sv;
        const float *rows = noise ? noise + (size_t)b * batch_size * t->num_children[t->root_id] : NULL;
        rc = select_batch(t, game, batch_size, coef, forced_k, noise_scale, rows, mix, lv);
        if (rc < 0)
            goto done;
        eval_stub(lv, game->n, stub_mode, value, prior, stride);
        rc = omcts_expand_backup(t, lv, value, prior, stride, &sv);
        if (rc < 0)
            goto done;
        sv_total += sv;
    }
    rc = 0;
    if (search_value)
        *search_value = sv_total / (float)(num_batches * batch_size);
done:
    free(lv);
    free(prior);
    return rc;
}

int omcts_sample_paths_stub_forced(otree *t, const ohex *game,
                                   int num_simulations, int batch_size,
                                   float coef, float forced_k, int stub_mode,
                                   float *search_value)
{
    return sample_paths_stub(t, game, num_simulations, batch_size, coef, forced_k, 0.0, NULL,
                             OMIX_F64, stub_mode, search_value);
}

int omcts_sample_paths_stub_noise(otree *t, const ohex *game,
                                  int num_simulations, int batch_size,
                                  float coef, float forced_k, double noise_scale,
                                  const float *noise, int mix, int stub_mode,
                                  float *search_value)
{
    return sample_paths_stub(t, game, num_simulations, batch_size, coef, forced_k, noise_scale,
                             noise, mix, stub_mode, search_value);
}
