"""The two training loops of the reference's `main.py` that drive the LSTUR path — `train` (main.py:56-96, the
`task/paper.py` handlers) and `cook` (main.py:147-297, the `Cook` handler) — as plain functions of a `settings.Config`.

The click command line itself is out of scope (DESIGN.md §8); what a caller of the path needs is the sequence of model
calls the commands make and the evaluation lines they log, reproduced here call for call:

    train:  for epoch: model = h.build_model(epoch); model.fit_generator(h.train, h.training_step, epochs=epoch + 1,
            initial_epoch=epoch); h.callback(epoch); model.evaluate_generator(h.valid, h.validation_step);
            h.callback_valid(epoch) ... h.save_model()
    cook:   for epoch: model = h.build_model(epoch); model.fit(*h.train(), batch_size, epochs=epoch + 1,
            initial_epoch=epoch, shuffle=True); h.callback(epoch); h.test_model.evaluate(*h.valid(), batch_size);
            h.callback_valid(epoch) ... then the per-user / per-impression / in-vocabulary / out-of-vocabulary averages of the
            scored test set (mnexp_b200/evaluation.py)

Both return the list of everything the reference would have logged through utils.logging_history /
utils.logging_evaluation, as ('history' | 'evaluation', dict) pairs in order (tests/test_ref_pinned.py compares that list
with the one the reference's own main.py produced).
"""
import logging

from . import evaluation, task, utils


class _Log:
    def __init__(self):
        self.records = []

    def history(self, history):
        self.records.append(('history', {k: list(v) for k, v in history.history.items()}))
        utils.logging_history(history)

    def evaluation(self, d):
        self.records.append(('evaluation', dict(d)))
        utils.logging_evaluation(d)


def _with_captured_evaluations(log, fn, *args):
    """handlers log their own evaluation lines through utils.logging_evaluation (task/paper.py:513-521): record those too"""
    orig = utils.logging_evaluation

    def tee(d):
        log.records.append(('evaluation', dict(d)))
        orig(d)
    utils.logging_evaluation = tee
    try:
        return fn(*args)
    finally:
        utils.logging_evaluation = orig


def train(config, on_build=None, device_batches=False, device_eval=False):
    """main.py:56-96.  on_build(handler) runs once after the first build_model (tests load reference weights there).
    device_batches: feed the handler's device_train / device_valid (batches assembled on the GPU, softmax-family handlers;
    their sampling differs from the host generators', mnexp_b200/assemble.py) where the loop feeds train / valid.
    device_eval: call handler.device_callback (the same impressions ranked on the GPU; the metrics differ by rounding
    only) where the loop calls handler.callback; independent of device_batches."""
    log = _Log()
    handler = task.get(config)
    if device_batches and not hasattr(handler, 'device_train'):
        raise NotImplementedError('%s has no device-assembled batches (the softmax-family handlers have)' % config.task)
    if device_eval and not getattr(handler, 'DEVICE_EVAL', False):
        raise NotImplementedError('%s has no device evaluation (the softmax-family handlers but ...VertAlt have)' % config.task)
    callback = getattr(handler, 'device_callback' if device_eval else 'callback', None)
    training_data = handler.device_train if device_batches else handler.train
    for epoch in range(config.epochs):
        logging.info('[+] start epoch {}'.format(epoch))
        model = handler.build_model(epoch)
        if epoch == 0 and on_build is not None:
            on_build(handler)
        history = model.fit_generator(training_data, handler.training_step, epochs=epoch + 1, initial_epoch=epoch, verbose=2)
        log.history(history)
        if callback is not None:
            _with_captured_evaluations(log, callback, epoch)
        try:
            valid = handler.device_valid if device_batches else handler.valid
            evaluations = model.evaluate_generator(valid, handler.validation_step, verbose=2)
            log.evaluation(dict(zip(model.metrics_names, evaluations)))
        except Exception:           # the reference swallows evaluation failures the same way (main.py:82-88)
            pass
        if hasattr(handler, 'callback_valid'):
            handler.callback_valid(epoch)
        logging.info('[-] finish epoch {}'.format(epoch))
    handler.save_model()
    return handler, log.records


def cook(config, on_build=None):
    """main.py:147-297 (the non-generator branch the reference's Cook handler supports)."""
    log = _Log()
    handler = task.get(config)
    for epoch in range(config.epochs):
        logging.info('[+] start epoch {}'.format(epoch))
        model = handler.build_model(epoch)
        if epoch == 0 and on_build is not None:
            on_build(handler)
        history = model.fit(*handler.train(), config.batch_size, epochs=epoch + 1, initial_epoch=epoch, shuffle=True, verbose=2)
        log.history(history)
        if hasattr(handler, 'callback'):
            _with_captured_evaluations(log, handler.callback, epoch)
        try:
            evaluations = handler.test_model.evaluate(*handler.valid(), config.batch_size, verbose=0)
            log.evaluation(dict(zip(handler.test_model.metrics_names, evaluations)))
        except Exception as e:
            print(e)
        if hasattr(handler, 'callback_valid'):
            handler.callback_valid(epoch)
        logging.info('[-] finish epoch {}'.format(epoch))
    feature, (users, imprs, mask, y_true) = handler.test()
    y_pred = handler.test_model.predict(feature, batch_size=config.batch_size, verbose=0).reshape((-1,))
    res = evaluation.aggregate(users, imprs, mask.reshape(-1), y_true, y_pred)
    evaluation.log_aggregate(res, log.evaluation)
    return handler, log.records
